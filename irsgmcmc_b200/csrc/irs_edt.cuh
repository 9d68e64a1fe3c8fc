// irs_edt.cuh -- the arithmetic of one line of the exact separable Euclidean distance transform (irs_surface.cu).
//
// Squared distances are carried in fp32 and weighted per axis by w = spacing^2.  With unit or dyadic spacings (1, 1.5, 2, ...)
// every value f + w k^2 the passes form is exactly representable below 2^24, so the transform is exact; otherwise each
// value carries fp32 rounding only.  __host__ __device__ so that the CPU tests run the very same code against brute force.
#pragma once
#include "irs_common.cuh"

// Pass 1, along a row: on entry d[i * ds] = 0 at the sites and +inf elsewhere; on exit the weighted squared distance
// w (i - j)^2 to the nearest site j (two sweeps).  A row without sites stays +inf.  Needs w > 0: a site is recognised by
// its 0, which no other element can hold.
IRS_HD void irs_edt_sites_1d(float* d, long long ds, int n, float w) {
    int last = -1;
    for (int i = 0; i < n; ++i) {
        if (d[i * ds] == 0.0f) last = i;
        else if (last >= 0) d[i * ds] = w * (float)((i - last) * (i - last));
    }
    int next = -1;
    for (int i = n - 1; i >= 0; --i) {
        const float v = d[i * ds];
        if (v == 0.0f) next = i;
        else if (next >= 0) d[i * ds] = fminf(v, w * (float)((next - i) * (next - i)));
    }
}

// Passes 2 and 3: d[i] <- min_j d[j] + w (i - j)^2 in place, as the lower envelope of parabolas (Felzenszwalb & Huttenlocher,
// "Distance Transforms of Sampled Functions", linear time).  Elements at +inf take no part; a line without a finite element
// stays +inf.  Scratch: v (n ints: apex positions), fv (n floats: their values, so that d can be overwritten), zb (n floats:
// left boundary of each parabola's interval), each element k at [k * ss].
IRS_HD void irs_edt_envelope_1d(float* d, long long ds, int n, float w, int* v, float* fv, float* zb, int ss) {
    int k = -1;
    for (int q = 0; q < n; ++q) {
        const float f = d[q * ds];
        if (!(f < INFINITY)) continue;
        const float hq = f + w * (float)(q * q);
        float s = -INFINITY;
        while (k >= 0) {
            const int p = v[k * ss];
            s = (hq - (fv[k * ss] + w * (float)(p * p))) / (2.0f * w * (float)(q - p));
            if (k > 0 && s <= zb[k * ss]) --k;   // parabola k is hidden under its neighbours: drop it
            else break;
        }
        ++k;
        v[k * ss] = q;
        fv[k * ss] = f;
        zb[k * ss] = s;
    }
    if (k < 0) return;
    const int K = k;
    k = 0;
    for (int q = 0; q < n; ++q) {
        while (k < K && zb[(k + 1) * ss] < (float)q) ++k;
        const int p = v[k * ss];
        d[q * ds] = fv[k * ss] + w * (float)((q - p) * (q - p));
    }
}
