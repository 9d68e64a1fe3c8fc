// irs_diagnostics.cu -- convergence diagnostics of the SGLD chains: voxel-wise split R-hat (Gelman et al., BDA3 section 11.4).
//   update   per kept sample, chain c's displacement (3,V) and warped image (1,V) folded into chain c's Welford (mean, M2) of
//            the current half of its kept samples (the first and last floor(N/2); the middle one of an odd N is skipped by the
//            caller).  Each (chain, half) is one sequence of the split R-hat.
//   sums     per element, over this GPU's sequences in index order (fp64): S1 = sum_j mean_j, SW = sum_j M2_j / (n - 1)
//   between  per element, against the grand mean S1 / M of ALL sequences: SB = sum_j (mean_j - S1 / M)^2
//   finish   R-hat = sqrt(var+ / W), W = SW / M, var+ = (n - 1) / n W + SB / (M - 1); summaries over the fixed mask by block
//            partials added up in a fixed order (no float atomics)
// With several GPUs, S1 / SW and then SB are sum-all-reduced between the phases (irsgmcmc_b200/parallel.py).
#include <cstdint>

#include "irs_kernels.cuh"

namespace {

// one sample of every chain: element e < 3V of chain c is disp[c][e], the rest im[c][e - 3V].  (mean, m2): (2, C, 4V).
// Same recurrence and operation order as welford_vec_kernel (irs_sampler.cu) with one new sample.
__global__ void __launch_bounds__(256)
split_welford_vec_kernel(const float* __restrict__ disp, const float* __restrict__ im, long long V, int C, int half,
                         double count, float* __restrict__ mean, float* __restrict__ m2) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // float4 index within the chain's 4V elements
    if (q >= V) return;
    const int c = blockIdx.y;
    const long long e = q * 4;
    const float* src = e < 3 * V ? disp + (size_t)c * 3 * V + e : im + (size_t)c * V + (e - 3 * V);
    const size_t o = ((size_t)half * C + c) * 4 * V + e;
    const float4 x = __ldg(reinterpret_cast<const float4*>(src));
    float4 m = *reinterpret_cast<const float4*>(mean + o), s = *reinterpret_cast<const float4*>(m2 + o);
    float cnt = (float)count;
    cnt += 1.f;
    float d;
    d = x.x - m.x; m.x += d / cnt; s.x += d * (x.x - m.x);
    d = x.y - m.y; m.y += d / cnt; s.y += d * (x.y - m.y);
    d = x.z - m.z; m.z += d / cnt; s.z += d * (x.z - m.z);
    d = x.w - m.w; m.w += d / cnt; s.w += d * (x.w - m.w);
    *reinterpret_cast<float4*>(mean + o) = m;
    *reinterpret_cast<float4*>(m2 + o) = s;
}

// the same for volumes whose size is not a multiple of 4 (or unaligned buffers)
__global__ void __launch_bounds__(256)
split_welford_kernel(const float* __restrict__ disp, const float* __restrict__ im, long long V, int C, int half,
                     double count, float* __restrict__ mean, float* __restrict__ m2) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= 4 * V) return;
    const int c = blockIdx.y;
    const float x = e < 3 * V ? disp[(size_t)c * 3 * V + e] : im[(size_t)c * V + (e - 3 * V)];
    const size_t o = ((size_t)half * C + c) * 4 * V + e;
    float m = mean[o], s = m2[o];
    float cnt = (float)count;
    cnt += 1.f;
    const float d = x - m;
    m += d / cnt;
    s += d * (x - m);
    mean[o] = m;
    m2[o] = s;
}

__global__ void __launch_bounds__(256)
split_rhat_sums_kernel(const float* __restrict__ mean, const float* __restrict__ m2, int n_seq, long long E, double nm1,
                       double* __restrict__ sums) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
        double s1 = 0.0, sw = 0.0;
#pragma unroll 4
        for (int j = 0; j < n_seq; ++j) {
            s1 += (double)__ldg(mean + (size_t)j * E + e);
            sw += (double)__ldg(m2 + (size_t)j * E + e) / nm1;
        }
        sums[e] = s1;
        sums[E + e] = sw;
    }
}

__global__ void __launch_bounds__(256)
split_rhat_between_kernel(const float* __restrict__ mean, int n_seq, long long E, const double* __restrict__ s1, double M,
                          double* __restrict__ sb) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (long long)gridDim.x * blockDim.x) {
        const double g = s1[e] / M;
        double s = 0.0;
#pragma unroll 4
        for (int j = 0; j < n_seq; ++j) {
            const double d = (double)__ldg(mean + (size_t)j * E + e) - g;
            s += d * d;
        }
        sb[e] = s;
    }
}

// W = 0 and B = 0 (every draw identical): 1;  W = 0 < B: +inf  (irsgmcmc_b200/utils/diagnostics.py:split_rhat has the same rules)
__device__ __forceinline__ float rhat_from_sums(double sw, double sb, int M, int n) {
    const double W = sw / M;
    if (W == 0.0) return sb == 0.0 ? 1.0f : INFINITY;
    const double var_plus = (double)(n - 1) / n * W + sb / (M - 1);
    return (float)sqrt(var_plus / W);
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// grid (blocks, n_comp): component k = blockIdx.y.  summary[k] = (max R-hat in the mask, voxels > 1.01, voxels > 1.1)
__global__ void __launch_bounds__(256)
split_rhat_finish_kernel(const double* __restrict__ sw, const double* __restrict__ sb, int M, int n,
                         const unsigned char* __restrict__ mask, long long V, float* __restrict__ rhat,
                         double* __restrict__ partials, unsigned int* __restrict__ counters, double* __restrict__ summary) {
    __shared__ double sh[3 * 8];
    __shared__ bool last;
    const int k = blockIdx.y, nb = gridDim.x;
    double mx = 0.0, c1 = 0.0, c2 = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)nb * blockDim.x) {
        const long long e = (long long)k * V + i;
        const float r = rhat_from_sums(sw[e], sb[e], M, n);
        rhat[e] = r;
        if (mask[i]) {
            mx = fmax(mx, (double)r);
            c1 += r > 1.01f ? 1.0 : 0.0;
            c2 += r > 1.1f ? 1.0 : 0.0;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    mx = warp_max(mx);
    c1 = irs_warp_sum(c1);
    c2 = irs_warp_sum(c2);
    if (lane == 0) { sh[warp] = mx; sh[8 + warp] = c1; sh[16 + warp] = c2; }
    __syncthreads();
    double* p = partials + (size_t)k * 3 * IRS_RHAT_REDUCE_BLOCKS;
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0, c = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a = fmax(a, sh[w]); b += sh[8 + w]; c += sh[16 + w]; }
        p[blockIdx.x] = a;
        p[IRS_RHAT_REDUCE_BLOCKS + blockIdx.x] = b;
        p[2 * IRS_RHAT_REDUCE_BLOCKS + blockIdx.x] = c;
        __threadfence();
        last = atomicAdd(counters + k, 1u) == (unsigned)(nb - 1);
    }
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    __threadfence();
    double a = 0.0, b = 0.0, c = 0.0;
    for (int g = 0; g < nb; ++g) {
        a = fmax(a, __ldcg(p + g));
        b += __ldcg(p + IRS_RHAT_REDUCE_BLOCKS + g);
        c += __ldcg(p + 2 * IRS_RHAT_REDUCE_BLOCKS + g);
    }
    summary[k * 3 + 0] = a;
    summary[k * 3 + 1] = b;
    summary[k * 3 + 2] = c;
    counters[k] = 0u;
}

unsigned grid_for(long long n) {
    const long long b = (n + 255) / 256;
    return (unsigned)(b < 148 * 8 ? b : 148 * 8);
}

}  // namespace

extern "C" int irs_split_welford_update(const float* disp, const float* im, int C, long long V, int half,
                                        double count_before, float* mean, float* m2, void* stream) {
    if (!disp || !im || !mean || !m2 || C < 1 || C > 65535 || V < 1 || (half != 0 && half != 1) || !(count_before >= 0))
        return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const bool vec = (V % 4) == 0 && ((reinterpret_cast<uintptr_t>(disp) | reinterpret_cast<uintptr_t>(im) |
                                       reinterpret_cast<uintptr_t>(mean) | reinterpret_cast<uintptr_t>(m2)) & 15) == 0;
    if (vec)
        split_welford_vec_kernel<<<dim3((unsigned)((V + 255) / 256), C), 256, 0, st>>>(disp, im, V, C, half, count_before,
                                                                                        mean, m2);
    else
        split_welford_kernel<<<dim3((unsigned)((4 * V + 255) / 256), C), 256, 0, st>>>(disp, im, V, C, half, count_before,
                                                                                        mean, m2);
    return (int)cudaGetLastError();
}

extern "C" int irs_split_rhat_sums(const float* mean, const float* m2, int n_seq, long long E, int n, double* sums,
                                   void* stream) {
    if (!mean || !m2 || !sums || n_seq < 1 || E < 1 || n < 2) return IRS_ERR_BAD_ARG;
    split_rhat_sums_kernel<<<grid_for(E), 256, 0, (cudaStream_t)stream>>>(mean, m2, n_seq, E, (double)(n - 1), sums);
    return (int)cudaGetLastError();
}

extern "C" int irs_split_rhat_between(const float* mean, int n_seq, long long E, const double* s1, int M, double* sb,
                                      void* stream) {
    if (!mean || !s1 || !sb || n_seq < 1 || E < 1 || M < 2 || n_seq > M) return IRS_ERR_BAD_ARG;
    split_rhat_between_kernel<<<grid_for(E), 256, 0, (cudaStream_t)stream>>>(mean, n_seq, E, s1, (double)M, sb);
    return (int)cudaGetLastError();
}

extern "C" int irs_split_rhat_finish(const double* sw, const double* sb, int M, int n, const unsigned char* mask, int n_comp,
                                     long long V, float* rhat, double* partials, unsigned int* counters, double* summary,
                                     void* stream) {
    if (!sw || !sb || !mask || !rhat || !partials || !counters || !summary || M < 2 || n < 2 || n_comp < 1 ||
        n_comp > IRS_RHAT_MAX_COMPONENTS || V < 1)
        return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(unsigned int) * n_comp, st);
    if (e != cudaSuccess) return (int)e;
    const long long b = (V + 255) / 256;
    const unsigned nb = (unsigned)(b < IRS_RHAT_REDUCE_BLOCKS ? b : IRS_RHAT_REDUCE_BLOCKS);
    split_rhat_finish_kernel<<<dim3(nb, n_comp), 256, 0, st>>>(sw, sb, M, n, mask, V, rhat, partials, counters, summary);
    return (int)cudaGetLastError();
}
