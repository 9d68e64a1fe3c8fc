// irs_select.cuh -- the arithmetic of the Hausdorff distance and its percentile (irs_surface.cu): which ranks of the directed
// distances a percentile reads, the digit step of the radix select over fp32 bit patterns, and numpy's linear interpolation.
//
// The keys are squared distances: non-negative and finite, so their fp32 bit patterns sort as their values do, and the square
// root (monotone) commutes with every order statistic.  Selection runs on the keys; the two selected keys are then taken to fp64,
// square-rooted and interpolated there.  __host__ __device__ so that the CPU tests run the very same code against np.percentile;
// irs_percentile_of_keys is the serial host restatement of hd_select_kernel's passes.
#pragma once
#include <math.h>
#include <string.h>

#include "irs_common.cuh"

#define IRS_SELECT_BITS 8                        // digit of one radix pass, most significant first
#define IRS_SELECT_BINS (1 << IRS_SELECT_BITS)
#define IRS_SELECT_PASSES (32 / IRS_SELECT_BITS)

// numpy.percentile(x, q) with its default method 'linear' over n sorted values s: h = (n - 1) (q / 100) in fp64; h >= n - 1 reads
// s[n - 1] alone (last), otherwise s[i] and s[i + 1] with i = floor(h), weight g = h - i
struct IrsPercentileRank {
    unsigned int i;
    double g;
    bool last;
};

IRS_HD IrsPercentileRank irs_percentile_rank(unsigned int n, double q) {
    const double h = (double)(n - 1) * (q / 100.0);
    IrsPercentileRank r;
    if (h >= (double)(n - 1)) {
        r.i = n - 1;
        r.g = 0.0;
        r.last = true;
    } else {
        r.i = (unsigned int)floor(h);
        r.g = h - (double)r.i;
        r.last = false;
    }
    return r;
}

// fp64 products and sums without contraction into an FMA: numpy rounds each operation on its own
IRS_HD double irs_mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}

IRS_HD double irs_add_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// the percentile of the distances from the squared distances at ranks i (lo) and i + 1 (hi; unused when last): numpy's _lerp,
// a + (b - a) g below g = 0.5 and b - (b - a) (1 - g) from there on
IRS_HD double irs_percentile_value(float lo, float hi, IrsPercentileRank r) {
    const double a = sqrt((double)lo);
    if (r.last) return a;
    const double b = sqrt((double)hi);
    const double d = irs_add_rn(b, -a);
    return r.g < 0.5 ? irs_add_rn(a, irs_mul_rn(d, r.g)) : irs_add_rn(b, -irs_mul_rn(d, irs_add_rn(1.0, -r.g)));
}

// one digit of a radix select: the first of the n bins whose cumulative count exceeds the rank r; r becomes the rank inside it
IRS_HD int irs_select_bin(const unsigned int* hist, int n, unsigned int* r) {
    for (int k = 0; k < n; ++k) {
        if (*r < hist[k]) return k;
        *r -= hist[k];
    }
    return n - 1;   // not reached for r < the sum of the bins
}

// host restatement of hd_select_kernel for one list of n >= 1 keys: the MSB-first digit passes for rank i, rank i + 1 as the same
// key when more than i + 1 keys are <= it and as the smallest key above it otherwise, then irs_percentile_value
inline double irs_percentile_of_keys(const float* keys, unsigned int n, double q) {
    const IrsPercentileRank pr = irs_percentile_rank(n, q);
    const unsigned int* bits = reinterpret_cast<const unsigned int*>(keys);
    unsigned int prefix = 0, mask = 0, r = pr.i, eq = 0;
    unsigned int hist[IRS_SELECT_BINS];
    for (int shift = 32 - IRS_SELECT_BITS; shift >= 0; shift -= IRS_SELECT_BITS) {
        for (int k = 0; k < IRS_SELECT_BINS; ++k) hist[k] = 0;
        for (unsigned int k = 0; k < n; ++k)
            if ((bits[k] & mask) == prefix) ++hist[(bits[k] >> shift) & (IRS_SELECT_BINS - 1)];
        const int bin = irs_select_bin(hist, IRS_SELECT_BINS, &r);
        eq = hist[bin];
        prefix |= (unsigned int)bin << shift;
        mask |= (unsigned int)(IRS_SELECT_BINS - 1) << shift;
    }
    unsigned int next = prefix;
    if (!pr.last && pr.i + 1 >= pr.i - r + eq) {   // keys <= rank i's key: (i - r) below it, eq equal to it
        next = 0xffffffffu;
        for (unsigned int k = 0; k < n; ++k)
            if (bits[k] > prefix && bits[k] < next) next = bits[k];
    }
    float lo, hi;
    memcpy(&lo, &prefix, 4);
    memcpy(&hi, &next, 4);
    return irs_percentile_value(lo, hi, pr);
}
