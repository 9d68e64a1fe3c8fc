// irs_landmark.cuh -- the per-landmark arithmetic of the landmark registration error and the landmark posterior
// (irs_landmark.cu): the predicted moving position of a fixed landmark, its TRE, the Welford step of the accumulators, and the
// finish (covariance, its eigenvalues, the squared Mahalanobis distance of the true position).
//
// Every fp64 product and sum goes through irs_mul_rn / irs_add_rn (irs_select.cuh), so nothing is contracted into an FMA: the
// device, a host build of this header and a numpy restatement that rounds each operation round the same way, and the predicted
// positions and TREs are bit-equal between them.  __host__ __device__ so that the CPU tests run this very code.
#pragma once
#include <math.h>

#include "../../include/irsgmcmc.h"   // IRS_LANDMARK_ACC, IRS_LANDMARK_COLS: the accumulator and posterior layouts
#include "irs_select.cuh"

// base index i0 = min(floor(p), n - 2), clamped to [0, n - 2] so that no coordinate (NaN or inf included) reads outside the
// volume; f = p - i0, which is p's fraction in [0, 1] for p in [0, n - 1]
IRS_HD int irs_landmark_base(double p, int n, double* f) {
    const double fl = floor(p);
    const int i0 = fl >= 0.0 ? (fl <= (double)(n - 2) ? (int)fl : n - 2) : 0;   // NaN compares false: 0
    *f = irs_add_rn(p, -(double)i0);
    return i0;
}

IRS_HD double irs_landmark_lerp(double a, double b, double f) { return irs_add_rn(a, irs_mul_rn(f, irs_add_rn(b, -a))); }

// predicted position m (moving voxel units, x y z) of the fixed landmark p (x y z) under one chain's normalised
// transformation T (3,D,H,W): trilinear interpolation in fp64 of the fp32 corners, lerps along x, then y, then z, and
// m_a = ((g_a + 1) (n_a - 1)) 0.5
IRS_HD void irs_landmark_predict(const float* T, int D, int H, int W, const double* p, double* m) {
    double fx, fy, fz;
    const int x0 = irs_landmark_base(p[0], W, &fx);
    const int y0 = irs_landmark_base(p[1], H, &fy);
    const int z0 = irs_landmark_base(p[2], D, &fz);
    const long long V = (long long)D * H * W, sy = W, sz = (long long)W * H;
    const long long b = (long long)z0 * sz + (long long)y0 * sy + x0;
    const int n[3] = {W, H, D};
    for (int ch = 0; ch < 3; ++ch) {
        const float* t = T + (size_t)ch * V + b;
        const double c00 = irs_landmark_lerp((double)t[0], (double)t[1], fx);
        const double c10 = irs_landmark_lerp((double)t[sy], (double)t[sy + 1], fx);
        const double c01 = irs_landmark_lerp((double)t[sz], (double)t[sz + 1], fx);
        const double c11 = irs_landmark_lerp((double)t[sz + sy], (double)t[sz + sy + 1], fx);
        const double c0 = irs_landmark_lerp(c00, c10, fy), c1 = irs_landmark_lerp(c01, c11, fy);
        const double g = irs_landmark_lerp(c0, c1, fz);
        m[ch] = irs_mul_rn(irs_mul_rn(irs_add_rn(g, 1.0), (double)(n[ch] - 1)), 0.5);
    }
}

// |s o (m - q)| in mm, the squares summed in x, y, z order
IRS_HD double irs_landmark_tre(const double* m, const double* q, const double* s) {
    double acc = 0.0;
    for (int a = 0; a < 3; ++a) {
        const double d = irs_mul_rn(s[a], irs_add_rn(m[a], -q[a]));
        acc = irs_add_rn(acc, irs_mul_rn(d, d));
    }
    return sqrt(acc);
}

// one Welford step with k = the count including this sample: delta = m - mean_old, mean += delta / k,
// M_ab += delta_a (m_b - mean_new,b) over (xx, xy, xz, yy, yz, zz); the TRE's mean and M2 the same way
IRS_HD void irs_landmark_welford(double* acc, double k, const double* m, double tre) {
    double d[3], e[3];
    for (int a = 0; a < 3; ++a) {
        d[a] = irs_add_rn(m[a], -acc[a]);
        acc[a] = irs_add_rn(acc[a], d[a] / k);
        e[a] = irs_add_rn(m[a], -acc[a]);
    }
    int j = 3;
    for (int a = 0; a < 3; ++a)
        for (int b = a; b < 3; ++b, ++j) acc[j] = irs_add_rn(acc[j], irs_mul_rn(d[a], e[b]));
    const double dt = irs_add_rn(tre, -acc[9]);
    acc[9] = irs_add_rn(acc[9], dt / k);
    acc[10] = irs_add_rn(acc[10], irs_mul_rn(dt, irs_add_rn(tre, -acc[9])));
}

// eigenvalues of a symmetric 2x2 [[a, b], [b, d]], larger first: mean +- hypot((a - d) / 2, b), no cancellation of close roots
IRS_HD void irs_sym2_eigen(double a, double b, double d, double* hi, double* lo) {
    const double m = 0.5 * (a + d), r = hypot(0.5 * (a - d), b);
    *hi = m + r;
    *lo = m - r;
}

// eigenvalues of the symmetric 3x3 (xx, xy, xz, yy, yz, zz) in descending order.  The trigonometric closed form of the
// characteristic cubic gives the eigenvalue that is farthest from the other two (the largest when the two smaller ones are the
// closer pair, else the smallest) to within a few ulps of the norm; its eigenvector (the largest cross product of two rows of
// A - lambda I) spans the complement in which the 2x2 projection gives the close pair without the sqrt(eps) loss the cubic has
// for them.  A diagonal matrix is sorted as it is.
IRS_HD void irs_sym3_eigen(const double* S, double* ev) {
    const double a = S[0], b = S[1], c = S[2], d = S[3], e = S[4], f = S[5];
    const double p1 = b * b + c * c + e * e;
    if (p1 == 0.0) {
        double x = a, y = d, z = f, t;
        if (x < y) { t = x; x = y; y = t; }
        if (y < z) { t = y; y = z; z = t; }
        if (x < y) { t = x; x = y; y = t; }
        ev[0] = x; ev[1] = y; ev[2] = z;
        return;
    }
    const double q = (a + d + f) / 3.0;
    const double aq = a - q, dq = d - q, fq = f - q;
    const double p = sqrt((aq * aq + dq * dq + fq * fq + 2.0 * p1) / 6.0);
    // det((A - q I) / p) / 2
    const double r0 = (aq * (dq * fq - e * e) - b * (b * fq - e * c) + c * (b * e - dq * c)) / (2.0 * p * p * p);
    const double r = r0 <= -1.0 ? -1.0 : (r0 >= 1.0 ? 1.0 : r0);
    const double phi = acos(r) / 3.0;
    const double pi23 = 2.0943951023931954923;   // 2 pi / 3
    const bool top = phi < 0.25 * pi23;           // phi < pi / 6: the largest is the isolated one
    const double lam = top ? q + 2.0 * p * cos(phi) : q + 2.0 * p * cos(phi + pi23);
    // eigenvector of lam: the largest of the three cross products of the rows (a - lam, b, c), (b, d - lam, e), (c, e, f - lam)
    const double al = a - lam, dl = d - lam, fl = f - lam;
    double v[3] = {b * e - c * dl, c * b - al * e, al * dl - b * b};   // row 1 x row 2
    double best = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
    const double x13[3] = {b * fl - c * e, c * c - al * fl, al * e - b * c};   // row 1 x row 3
    const double n13 = x13[0] * x13[0] + x13[1] * x13[1] + x13[2] * x13[2];
    if (n13 > best) { best = n13; v[0] = x13[0]; v[1] = x13[1]; v[2] = x13[2]; }
    const double x23[3] = {dl * fl - e * e, e * c - b * fl, b * e - dl * c};   // row 2 x row 3
    const double n23 = x23[0] * x23[0] + x23[1] * x23[1] + x23[2] * x23[2];
    if (n23 > best) { best = n23; v[0] = x23[0]; v[1] = x23[1]; v[2] = x23[2]; }
    double lo_pair, hi_pair;
    if (!(best > 0.0)) {   // no usable direction (all three coincide to rounding): the spread is below the rounding level
        lo_pair = hi_pair = q;
    } else {
        const double inv = 1.0 / sqrt(best);
        v[0] *= inv; v[1] *= inv; v[2] *= inv;
        // orthonormal u, w completing v: u from the axis least aligned with v
        const double ax = fabs(v[0]), ay = fabs(v[1]), az = fabs(v[2]);
        double u[3];
        if (ax <= ay && ax <= az) { u[0] = 0.0; u[1] = v[2]; u[2] = -v[1]; }
        else if (ay <= az) { u[0] = -v[2]; u[1] = 0.0; u[2] = v[0]; }
        else { u[0] = v[1]; u[1] = -v[0]; u[2] = 0.0; }
        const double un = 1.0 / sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
        u[0] *= un; u[1] *= un; u[2] *= un;
        const double w[3] = {v[1] * u[2] - v[2] * u[1], v[2] * u[0] - v[0] * u[2], v[0] * u[1] - v[1] * u[0]};
        const double Au[3] = {a * u[0] + b * u[1] + c * u[2], b * u[0] + d * u[1] + e * u[2], c * u[0] + e * u[1] + f * u[2]};
        const double Aw[3] = {a * w[0] + b * w[1] + c * w[2], b * w[0] + d * w[1] + e * w[2], c * w[0] + e * w[1] + f * w[2]};
        irs_sym2_eigen(u[0] * Au[0] + u[1] * Au[1] + u[2] * Au[2], u[0] * Aw[0] + u[1] * Aw[1] + u[2] * Aw[2],
                       w[0] * Aw[0] + w[1] * Aw[1] + w[2] * Aw[2], &hi_pair, &lo_pair);
    }
    if (top) { ev[0] = lam; ev[1] = hi_pair; ev[2] = lo_pair; }
    else { ev[0] = hi_pair; ev[1] = lo_pair; ev[2] = lam; }
    // the pair and the isolated eigenvalue come from different formulas: sort the three where rounding crossed them
    if (ev[1] > ev[0]) { const double t = ev[0]; ev[0] = ev[1]; ev[1] = t; }
    if (ev[2] > ev[1]) { const double t = ev[1]; ev[1] = ev[2]; ev[2] = t; }
    if (ev[1] > ev[0]) { const double t = ev[0]; ev[0] = ev[1]; ev[1] = t; }
}

// r^T S^-1 r by the Cholesky factor of S (xx, xy, xz, yy, yz, zz), factorised and solved in a fixed order; a pivot <= 0
// (or NaN) gives +inf
IRS_HD double irs_sym3_mahalanobis2(const double* S, const double* r) {
    const double inf = (double)INFINITY;
    if (!(S[0] > 0.0)) return inf;
    const double l00 = sqrt(S[0]);
    const double l10 = S[1] / l00, l20 = S[2] / l00;
    const double t11 = S[3] - l10 * l10;
    if (!(t11 > 0.0)) return inf;
    const double l11 = sqrt(t11);
    const double l21 = (S[4] - l20 * l10) / l11;
    const double t22 = S[5] - l20 * l20 - l21 * l21;
    if (!(t22 > 0.0)) return inf;
    const double l22 = sqrt(t22);
    const double y0 = r[0] / l00;
    const double y1 = (r[1] - l10 * y0) / l11;
    const double y2 = (r[2] - l20 * y0 - l21 * y1) / l22;
    return y0 * y0 + y1 * y1 + y2 * y2;
}

// the posterior row of one landmark from its accumulators over n >= 1 samples (layout in include/irsgmcmc.h):
// [0, 3) mean position (moving voxels), [3] TRE of the mean, [4] E[TRE], [5] std of TRE, [6, 12) covariance in mm^2,
// [12, 15) principal standard deviations (mm, descending), [15] squared Mahalanobis distance of q; [5, 16) NaN for n < 2
IRS_HD void irs_landmark_finish(const double* acc, double n, const double* q, const double* s, double* out) {
    out[0] = acc[0]; out[1] = acc[1]; out[2] = acc[2];
    out[3] = irs_landmark_tre(acc, q, s);
    out[4] = acc[9];
    if (!(n >= 2.0)) {
        for (int k = 5; k < IRS_LANDMARK_COLS; ++k) out[k] = (double)NAN;
        return;
    }
    const double nm1 = n - 1.0;
    out[5] = sqrt(acc[10] / nm1);
    double S[6];
    int j = 0;
    for (int a = 0; a < 3; ++a)
        for (int b = a; b < 3; ++b, ++j) S[j] = irs_mul_rn(irs_mul_rn(s[a], s[b]), acc[3 + j]) / nm1;
    for (int k = 0; k < 6; ++k) out[6 + k] = S[k];
    double ev[3];
    irs_sym3_eigen(S, ev);
    for (int k = 0; k < 3; ++k) out[12 + k] = sqrt(ev[k] > 0.0 ? ev[k] : 0.0);
    double r[3];
    for (int a = 0; a < 3; ++a) r[a] = irs_mul_rn(s[a], irs_add_rn(q[a], -acc[a]));
    out[15] = irs_sym3_mahalanobis2(S, r);
}
