// irs_landmark.cu -- landmark registration error and landmark posterior over every accumulated sample.
//   map        one thread per (chain, landmark): the predicted moving position of the fixed landmark under the chain's
//              transformation T and its TRE (irs_landmark_predict / irs_landmark_tre).
//   update     one launch per kept sample.  Blocks [0, tiles) own LM_BLOCK landmarks each, one per thread: a thread reads its
//              landmark's 11 accumulators once, folds the C chains in index order (irs_landmark_welford) and writes them back,
//              so splitting the chains of a sample over several launches gives the same bits.  Blocks [tiles, tiles + chain
//              blocks) own one chain per thread and add that chain's TREs in landmark order (sum, sum of squares, max).
//   posterior  one thread per landmark: irs_landmark_finish.
// No atomics, no host synchronisation, no dependency on scheduling.
#include "irs_kernels.cuh"
#include "irs_landmark.cuh"

namespace {

constexpr int LM_BLOCK = 128;

struct Spacing {
    double s[3];
};

__global__ void __launch_bounds__(LM_BLOCK)
landmark_map_kernel(const float* __restrict__ T, int C, int D, int H, int W, const double* __restrict__ p,
                    const double* __restrict__ q, int P, Spacing sp, double* __restrict__ pred, double* __restrict__ tre) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)C * P) return;
    const int c = (int)(t / P), i = (int)(t % P);
    const double pi[3] = {p[3 * i], p[3 * i + 1], p[3 * i + 2]};
    const double qi[3] = {q[3 * i], q[3 * i + 1], q[3 * i + 2]};
    double m[3];
    irs_landmark_predict(T + (size_t)c * 3 * D * H * W, D, H, W, pi, m);
    double* o = pred + 3 * t;
    o[0] = m[0]; o[1] = m[1]; o[2] = m[2];
    tre[t] = irs_landmark_tre(m, qi, sp.s);
}

__global__ void __launch_bounds__(LM_BLOCK)
landmark_update_kernel(const double* __restrict__ pred, const double* __restrict__ tre, int C, int P, int tiles,
                       double count_before, double* __restrict__ acc, double* __restrict__ sample_stats) {
    if ((int)blockIdx.x < tiles) {
        const int i = blockIdx.x * LM_BLOCK + threadIdx.x;
        if (i >= P) return;
        double a[IRS_LANDMARK_ACC];
        double* g = acc + (size_t)IRS_LANDMARK_ACC * i;
#pragma unroll
        for (int k = 0; k < IRS_LANDMARK_ACC; ++k) a[k] = g[k];
        for (int c = 0; c < C; ++c) {
            const size_t t = (size_t)c * P + i;
            const double m[3] = {__ldg(pred + 3 * t), __ldg(pred + 3 * t + 1), __ldg(pred + 3 * t + 2)};
            irs_landmark_welford(a, count_before + (double)(c + 1), m, __ldg(tre + t));
        }
#pragma unroll
        for (int k = 0; k < IRS_LANDMARK_ACC; ++k) g[k] = a[k];
        return;
    }
    const int c = ((int)blockIdx.x - tiles) * LM_BLOCK + threadIdx.x;
    if (c >= C) return;
    const double* r = tre + (size_t)c * P;
    double s = 0.0, s2 = 0.0, mx = 0.0;
    for (int i = 0; i < P; ++i) {
        const double x = __ldg(r + i);
        s = irs_add_rn(s, x);
        s2 = irs_add_rn(s2, irs_mul_rn(x, x));
        mx = i == 0 || x > mx || x != x ? x : mx;   // a NaN TRE (non-finite T) stays the maximum, as np.max has it
    }
    double* o = sample_stats + 3 * (size_t)c;
    o[0] = s; o[1] = s2; o[2] = mx;
}

__global__ void __launch_bounds__(LM_BLOCK)
landmark_posterior_kernel(const double* __restrict__ acc, const double* __restrict__ q, int P, double n, Spacing sp,
                          double* __restrict__ out) {
    const int i = blockIdx.x * LM_BLOCK + threadIdx.x;
    if (i >= P) return;
    double a[IRS_LANDMARK_ACC], o[IRS_LANDMARK_COLS];
#pragma unroll
    for (int k = 0; k < IRS_LANDMARK_ACC; ++k) a[k] = acc[(size_t)IRS_LANDMARK_ACC * i + k];
    const double qi[3] = {q[3 * i], q[3 * i + 1], q[3 * i + 2]};
    irs_landmark_finish(a, n, qi, sp.s, o);
#pragma unroll
    for (int k = 0; k < IRS_LANDMARK_COLS; ++k) out[(size_t)IRS_LANDMARK_COLS * i + k] = o[k];
}

bool spacing_ok(const double* s, Spacing* sp) {
    if (!s) return false;
    for (int a = 0; a < 3; ++a) {
        if (!(s[a] > 0.0) || !isfinite(s[a])) return false;
        sp->s[a] = s[a];
    }
    return true;
}

constexpr double TWO53 = 9007199254740992.0;

unsigned blocks(long long n) { return (unsigned)((n + LM_BLOCK - 1) / LM_BLOCK); }

}  // namespace

extern "C" int irs_landmark_map(const float* T, int C, int D, int H, int W, const double* p, const double* q, int P,
                                const double* spacing_host, double* pred, double* tre, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    Spacing sp;
    if (!T || !p || !q || !pred || !tre || P < 1 || !spacing_ok(spacing_host, &sp)) return IRS_ERR_BAD_ARG;
    if ((long long)C * P > 0x7fffffffLL) return IRS_ERR_UNSUPPORTED;
    landmark_map_kernel<<<blocks((long long)C * P), LM_BLOCK, 0, (cudaStream_t)stream>>>(T, C, D, H, W, p, q, P, sp, pred,
                                                                                         tre);
    return (int)cudaGetLastError();
}

extern "C" int irs_landmark_update(const double* pred, const double* tre, int C, int P, double count_before, double* acc,
                                   double* sample_stats, void* stream) {
    if (!pred || !tre || !acc || !sample_stats || C < 1 || P < 1 || !(count_before >= 0.0) ||
        count_before != floor(count_before) || count_before > TWO53 - (double)C)   // exact: C < 2^31
        return IRS_ERR_BAD_ARG;
    if ((long long)C * P > 0x7fffffffLL) return IRS_ERR_UNSUPPORTED;
    const int tiles = (int)blocks(P);
    landmark_update_kernel<<<tiles + blocks(C), LM_BLOCK, 0, (cudaStream_t)stream>>>(pred, tre, C, P, tiles, count_before,
                                                                                    acc, sample_stats);
    return (int)cudaGetLastError();
}

extern "C" int irs_landmark_posterior(const double* acc, const double* q, int P, long long n, const double* spacing_host,
                                      double* out, void* stream) {
    Spacing sp;
    if (!acc || !q || !out || P < 1 || n < 1 || n > (1LL << 53) || !spacing_ok(spacing_host, &sp)) return IRS_ERR_BAD_ARG;
    landmark_posterior_kernel<<<blocks(P), LM_BLOCK, 0, (cudaStream_t)stream>>>(acc, q, P, (double)n, sp, out);
    return (int)cudaGetLastError();
}
