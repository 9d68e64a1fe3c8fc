"""
fp64 references of the Langevin + Sobolev proposal and of the LCC box-filter passes, with per-voxel rounding bounds.

Each function takes the fp32 inputs the kernel itself read for that stage (for a later pass: the kernel's own output of
the earlier pass) and returns (out, bound), both fp64 and of the output's shape.  Stages are checked one at a time, so
errors never compound, and a kernel result must satisfy |kernel - out| <= bound on every voxel.  Given fp64 inputs the
functions compute the exact operations, which test_transition_ref.py checks against the oracle (oracle/sgld_oracle.py).

Neither stage takes a decision on a rounded value (no floor, no comparison), so nothing has to be emulated: every fp32
operation only rounds and is bounded.  The library is compiled without --use_fast_math, so sqrtf and 1.0f / x are
correctly rounded; a product may or may not be contracted into an FMA, and the bounds below hold either way.

Rounding bounds (u = 2^-24, first order; SO = 1 + 2^-10 covers the second-order terms: every m u below is < 2^-10)
--------------------------------------------------------------------------------------------------------------------
A filter pass out(j) = sum_t w_t x_t over NT taps, accumulated in fp32 from zero in any order, rounds each of the NT
products (when not contracted into an FMA) and each of the NT - 1 additions by at most u times the sum of the
magnitudes of its terms:

    pass rounding <= (2 NT - 1) u sum_t |w_t x_t| <= 2 NT u |W| |x|

where |W| is the pass applied with |w_t| (for the adjoint passes: the transpose with its fold weights).  An input error
b passes through a pass as |W| b.  The weights themselves are the fp32 values the kernel holds (the Sobolev taps as
host_floats rounds them), i.e. exact inputs; the box weights are small integers.

Langevin + Sobolev, out = S_x S_y S_z (v + coef sigma eps) with replicate padding (csrc/irs_smooth.cu):
  * proposal p = fl(v + fl(fl(coef sigma) eps)): the two products and the sum round, <= u (|v| + 3 |coef sigma eps|)
    (a contracted FMA only removes a rounding);
  * three passes in either order (the fused kernel runs x, y, z; the four-pass path z, y, x).  The taps are positive,
    so |S| = S and the magnitudes |S|^k |p| the passes see do not depend on the order.  Every pass adds 2 NT u S (..)
    of the magnitudes it sees, and the later passes carry it with S:

    |out_kernel - out| <= u SO S^3 ( |v| + 3 |coef sigma eps| + 6 NT (|p| + b_p) ),   b_p the proposal bound

LCC normalisation (csrc/irs_data.cu box_march_kernel: three box passes of 2 S + 1 ones, then an epilogue), k3 = (2S+1)^3
and inv_k3 = fl32(1 / k3) (relative error <= u); B(.) the replicate box sum, B^T its adjoint (fold weights at the faces):
  * FWD_MEAN  a = I - B(I) / k3.  The box sum rounds by <= 3 * 2 NT u B(|I|); the scale by inv_k3 and the product add
    2u |B(I)| / k3, the difference u |a|:
        |a_kernel - a| <= u SO ( |a| + (6 NT + 2) B(|I|) / k3 )
  * FWD_VAR   var = B(a^2) / k3 from the kernel's own a, rs = 1 / sqrt(var + 1e-10), z = zF - a rs (zF absent: a rs).
    All terms are positive, so every rounding is relative: a^2 (u), the box (6 NT u), inv_k3 and the product (2u), the
    sum with fl32(1e-10) (2u: the constant and the add); sqrt halves that and rounds (u), the division rounds (u):
        |rs_kernel - rs| <= u SO rs ( (6 NT + 5) / 2 + 2 ),   e_rs the relative bound in parentheses times u SO
        |z_kernel - z|   <= u SO ( |z| + |a rs| (1 + e_rs / (u SO)) )     (the product, the difference)
  * BWD_VAR   pre = -1/2 g a rs^3 (g = sign g_in; the factor -1/2 sign is exact, then four products round: 4u |pre|),
    ga = g rs + 2 a B^T(pre) / k3:
        |ga_kernel - ga| <= u SO ( |g rs| + |ga| + 2 |a| (6 NT + 2 + 4) B^T(|pre|) / k3 + 2 |a B^T(pre)| / k3 )
    (the two products and the sum of the epilogue, the adjoint box, inv_k3 and its product, the pre-operation)
  * BWD_MEAN  g_I = ga - B^T(ga) / k3 from the kernel's own ga:
        |g_kernel - g_I| <= u SO ( |g_I| + (6 NT + 2) B^T(|ga|) / k3 )
"""
import numpy as np
import torch

U24 = 2.0 ** -24
SO = 1.0 + 2.0 ** -10
AXES = (2, 3, 4)   # z, y, x of a (C, channels, D, H, W) tensor


def fp32_taps(taps):
    """the taps as the kernel holds them (host_floats rounds them to fp32)"""
    return [float(np.float32(t)) for t in taps]


# ---- separable passes with replicate padding ---------------------------------------------------------------------------
def _shift(x, axis, offset):
    n = x.shape[axis]
    idx = torch.clamp(torch.arange(n, device=x.device) + offset, 0, n - 1)
    return x.index_select(axis, idx)


def filter_axis(x, axis, weights):
    """out(j) = sum_t w_t x(clamp(j + t - s)), s = (len(weights) - 1) / 2"""
    s = (len(weights) - 1) // 2
    out = torch.zeros_like(x)
    for t, w in enumerate(weights):
        out = out + float(w) * _shift(x, axis, t - s)
    return out


def filter_axis_adjoint(x, axis, weights):
    """the transpose of filter_axis: every x(j) goes to clamp(j + t - s) with w_t, so a face collects the folded taps"""
    s = (len(weights) - 1) // 2
    n = x.shape[axis]
    out = torch.zeros_like(x)
    for t, w in enumerate(weights):
        idx = torch.clamp(torch.arange(n, device=x.device) + t - s, 0, n - 1)
        out.index_add_(axis, idx, float(w) * x)
    return out


def smooth3(x, weights, adjoint=False):
    f = filter_axis_adjoint if adjoint else filter_axis
    for axis in AXES:
        x = f(x, axis, weights)
    return x


# ---- Langevin proposal + Sobolev smoothing ----------------------------------------------------------------------------
def langevin_smooth(v, sigma, coef, eps, taps):
    """(out, bound) of S_x S_y S_z (v + coef sigma eps); sigma None = 1, broadcast over chains if its first dim is 1;
    taps as the caller passes them (rounded to fp32 here like the launcher does); coef = 0 ignores eps"""
    v = v.double()
    if coef == 0.0:
        noise = torch.zeros_like(v)
    else:
        sg = 1.0 if sigma is None else sigma.double()
        noise = float(np.float32(coef)) * sg * eps.double()
    p = v + noise
    b_p = U24 * (v.abs() + 3.0 * noise.abs())
    if not len(taps):
        return p, SO * b_p
    w = fp32_taps(taps)
    assert all(t >= 0 for t in w), 'the order-free bound needs positive taps'
    nt = len(w)
    out = smooth3(p, w)
    bound = SO * smooth3(b_p + 6 * nt * U24 * (p.abs() + b_p), w)
    return out, bound


# ---- LCC normalisation and its adjoint ---------------------------------------------------------------------------------
def _box(x, S, adjoint=False):
    return smooth3(x, [1.0] * (2 * S + 1), adjoint)


def lcc_fwd_mean(I, S):
    """(a, bound): a = I - B(I) / k3"""
    I = I.double()
    k3, nt = float((2 * S + 1) ** 3), 2 * S + 1
    a = I - _box(I, S) / k3
    return a, U24 * SO * (a.abs() + (6 * nt + 2) * _box(I.abs(), S) / k3)


def lcc_fwd_var(a, zF, S):
    """((rs, rs bound), (z, z bound)) from the kernel's own a: rs = 1 / sqrt(B(a^2) / k3 + 1e-10), z = zF - a rs or a rs"""
    a = a.double()
    k3, nt = float((2 * S + 1) ** 3), 2 * S + 1
    rs = 1.0 / torch.sqrt(_box(a * a, S) / k3 + 1e-10)
    e_rs = U24 * SO * ((6 * nt + 5) / 2.0 + 2.0)
    zn = a * rs
    z = zn if zF is None else zF.double() - zn
    b_z = U24 * SO * (z.abs() + zn.abs()) + zn.abs() * e_rs
    return (rs, e_rs * rs), (z, b_z)


def lcc_bwd_var(g, sign, a, rs, S):
    """(ga, bound): ga = g rs + 2 a B^T(-1/2 g a rs^3) / k3 with g = sign g_in, from the kernel's own a and rs"""
    g = float(sign) * g.double()
    a, rs = a.double(), rs.double()
    k3, nt = float((2 * S + 1) ** 3), 2 * S + 1
    pre = -0.5 * g * a * rs ** 3
    bt = _box(pre, S, adjoint=True) / k3
    ga = g * rs + 2.0 * a * bt
    mag = _box(pre.abs(), S, adjoint=True) / k3
    bound = U24 * SO * ((g * rs).abs() + ga.abs() + 2.0 * a.abs() * ((6 * nt + 6) * mag + bt.abs()))
    return ga, bound


def lcc_bwd_mean(ga, S):
    """(g_I, bound): g_I = ga - B^T(ga) / k3, from the kernel's own ga"""
    ga = ga.double()
    k3, nt = float((2 * S + 1) ** 3), 2 * S + 1
    gi = ga - _box(ga, S, adjoint=True) / k3
    return gi, U24 * SO * (gi.abs() + (6 * nt + 2) * _box(ga.abs(), S, adjoint=True) / k3)


def worst(out, ref, bound):
    """(number of voxels outside the bound, index of the worst one, its |difference| / bound, median ratio)"""
    d = (out.double() - ref.double()).abs()
    bad = ~(d <= bound)   # NaN counts as outside
    ratio = torch.where(bad & ~(d < float('inf')), float('inf'), d / bound.clamp_min(1e-300))
    i = int(torch.argmax(ratio))
    at = tuple(int(x) for x in torch.unravel_index(torch.tensor(i), out.shape))
    return int(bad.sum()), at, float(ratio.flatten()[i]), float(ratio.flatten().median())
