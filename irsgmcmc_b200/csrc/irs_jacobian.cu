// irs_jacobian.cu -- posterior of the Jacobian determinant of the transformation over every accumulated sample.
//   ld(c, v)  log det J of chain c's transformation T (C,3,D,H,W) in normalised units at voxel v, exactly as
//             irs_log_det_jacobian computes it: forward differences with the last one replicated, times (n - 1) / 2, the six
//             products in the reference's order, logf (irs_log_det_3x3).  A sample is finite at v when ld is finite (det > 0);
//             otherwise it is folded there: det < 0 (NaN, the reference's folding), det == 0 (-inf), NaN or inf input.
//   update    per kept sample, for all C chains in one launch: folds[v] += folded samples; (mean, m2)[v] = fp32 Welford of ld
//             over the finite samples only, with the recurrence and operation order of welford_vec_kernel (irs_sampler.cu) and
//             the running count starting at count_before - folds[v].  Each thread owns VW consecutive x voxels of one row and
//             loops over the chains with the next chain's loads in flight; the accumulators are read and written once.  Per
//             chain, over the fixed mask: (finite voxels, folded voxels, sum ld, sum ld^2) -- the counts through one 64-bit
//             integer atomicAdd per block and chunk of chains, the sums through block partials that the last block adds up in
//             a fixed order.  No float atomics: the result does not depend on scheduling.
//   finish    p_fold = (float)folds / (float)n; mean (NaN where n_v = n - folds = 0); std = sqrt(m2 / (n_v - 1)) (NaN where
//             n_v < 2); over the mask exact int64 sums (folds, voxels with folds > 0, voxels with 2 folds > n) and the fp64
//             means of the mean and std maps from fixed-order block partials.
#include <cstdint>

#include "irs_kernels.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int CHUNK = 32;   // chains whose per-block sums are gathered in shared memory between two block barriers

// one chain's values at this thread's VW voxels, components x, y, z.  VW = 4: the rows (z,y), (z,y+-1), (z+-1,y) as float4
// and the x + 1 neighbour of the fourth voxel (read by the last lane of a warp only; the others take it from the next lane).
// VW = 1: the six values of log_det_j_kernel's differences.
template <int VW>
struct ChainLoads;

template <>
struct ChainLoads<4> {
    float4 c[3], y[3], z[3];
    float xn[3];
    __device__ __forceinline__ void load(const float* __restrict__ t, long long V, long long i0, long long oy, long long oz,
                                         bool load_xn) {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* f = t + (size_t)ch * V + i0;
            c[ch] = __ldg(reinterpret_cast<const float4*>(f));
            y[ch] = __ldg(reinterpret_cast<const float4*>(f + oy));
            z[ch] = __ldg(reinterpret_cast<const float4*>(f + oz));
            xn[ch] = load_xn ? __ldg(f + 4) : 0.f;
        }
    }
};

template <>
struct ChainLoads<1> {
    float x0[3], x1[3], y0[3], y1[3], z0[3], z1[3];
    __device__ __forceinline__ void load(const float* __restrict__ t, long long V, long long ix, long long iy, long long iz,
                                         long long sy, long long sz) {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* f = t + (size_t)ch * V;
            x0[ch] = __ldg(f + ix); x1[ch] = __ldg(f + ix + 1);
            y0[ch] = __ldg(f + iy); y1[ch] = __ldg(f + iy + sy);
            z0[ch] = __ldg(f + iz); z1[ch] = __ldg(f + iz + sz);
        }
    }
};

__device__ __forceinline__ float elem(const float4& v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }

// grid-stride over groups of VW voxels (V % VW == 0 for VW = 4: W % 4 == 0); every thread of a block runs the same number of
// iterations and chains, so the warp shuffles and block barriers below see every thread.
// partials: [c][0] sum ld, [c][1] sum ld^2, gridDim.x doubles each; counters: C packed counts (folded << 32 | finite), then the
// ticket -- zero on entry, left zero.
template <int VW>
__global__ void __launch_bounds__(256)
jacobian_update_kernel(const float* __restrict__ T, const unsigned char* __restrict__ mask, int C, IrsDims d,
                       double count_before, int* __restrict__ folds, float* __restrict__ mean, float* __restrict__ m2,
                       double* __restrict__ partials, unsigned long long* __restrict__ counters,
                       double* __restrict__ sample_stats) {
    __shared__ double sh_s[CHUNK][8], sh_q[CHUNK][8];
    __shared__ unsigned sh_n[CHUNK][8];
    __shared__ bool last;
    const long long V = d.V();
    const long long sy = d.W, sz = (long long)d.W * d.H;
    const float kx = 0.5f * (float)(d.W - 1), ky = 0.5f * (float)(d.H - 1), kz = 0.5f * (float)(d.D - 1);
    const long long nq = V / VW;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = gridDim.x;
    int pass = 0;
    for (long long base = (long long)blockIdx.x * blockDim.x; base < nq; base += (long long)G * blockDim.x, ++pass) {
        const bool active = base + threadIdx.x < nq;
        const long long q = active ? base + threadIdx.x : nq - 1;   // inactive threads shadow the last group, write nothing
        const long long i0 = q * VW;
        const int x0 = (int)(i0 % d.W);
        const int y = (int)((i0 / d.W) % d.H), z = (int)(i0 / sz);
        const bool y_end = y == d.H - 1, z_end = z == d.D - 1;
        // VW = 4: the x + 1 neighbour of the fourth voxel exists unless it ends the row; the next lane holds it, except in lane 31
        const bool x_end = x0 + VW - 1 == d.W - 1;
        const bool load_xn = lane == 31 && !x_end;

        unsigned char mk[VW];
        int fo[VW];
        float mu[VW], s2[VW], cnt[VW];
        if constexpr (VW == 4) {
            const uchar4 m4 = *reinterpret_cast<const uchar4*>(mask + i0);
            const int4 f4 = *reinterpret_cast<const int4*>(folds + i0);
            const float4 a4 = *reinterpret_cast<const float4*>(mean + i0), b4 = *reinterpret_cast<const float4*>(m2 + i0);
            mk[0] = m4.x; mk[1] = m4.y; mk[2] = m4.z; mk[3] = m4.w;
            fo[0] = f4.x; fo[1] = f4.y; fo[2] = f4.z; fo[3] = f4.w;
            mu[0] = a4.x; mu[1] = a4.y; mu[2] = a4.z; mu[3] = a4.w;
            s2[0] = b4.x; s2[1] = b4.y; s2[2] = b4.z; s2[3] = b4.w;
        } else {
            mk[0] = mask[i0]; fo[0] = folds[i0]; mu[0] = mean[i0]; s2[0] = m2[i0];
        }
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            if (!active) mk[k] = 0;
            cnt[k] = (float)(count_before - (double)fo[k]);   // finite samples so far: welford_vec_kernel's (float)count
        }

        ChainLoads<VW> cur, nxt;
        long long a0, a1, a2;   // VW = 4: i0, row offsets;  VW = 1: ix, iy, iz of log_det_j_kernel
        if constexpr (VW == 4) {
            a0 = i0; a1 = y_end ? -sy : sy; a2 = z_end ? -sz : sz;
            cur.load(T, V, a0, a1, a2, load_xn);
        } else {
            a0 = x_end ? i0 - 1 : i0; a1 = y_end ? i0 - sy : i0; a2 = z_end ? i0 - sz : i0;
            cur.load(T, V, a0, a1, a2, sy, sz);
        }
        for (int c = 0; c < C; ++c) {
            if (c + 1 < C) {
                const float* t = T + (size_t)(c + 1) * 3 * V;
                if constexpr (VW == 4) nxt.load(t, V, a0, a1, a2, load_xn);
                else nxt.load(t, V, a0, a1, a2, sy, sz);
            }
            float xn[3];   // VW = 4: f(i0 + 4) of each component, from the next lane (its first voxel) or loaded by lane 31
            if constexpr (VW == 4) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    xn[ch] = __shfl_down_sync(FULL, cur.c[ch].x, 1);
                    if (lane == 31) xn[ch] = cur.xn[ch];
                }
            }
            double s = 0.0, sq = 0.0;
            unsigned n_fin = 0u, n_fold = 0u;
#pragma unroll
            for (int k = 0; k < VW; ++k) {
                float J[3][3];   // J[j][comp]
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    if constexpr (VW == 4) {
                        const float4& r = cur.c[ch];
                        float hi, lo;   // (f(ix + 1), f(ix)) with ix = i, or i - 1 at the end of the row
                        if (k < 3) { hi = elem(r, k + 1); lo = elem(r, k); }
                        else if (!x_end) { hi = xn[ch]; lo = r.w; }
                        else { hi = r.w; lo = r.z; }
                        J[0][ch] = (hi - lo) * kx;
                        J[1][ch] = (y_end ? elem(r, k) - elem(cur.y[ch], k) : elem(cur.y[ch], k) - elem(r, k)) * ky;
                        J[2][ch] = (z_end ? elem(r, k) - elem(cur.z[ch], k) : elem(cur.z[ch], k) - elem(r, k)) * kz;
                    } else {
                        J[0][ch] = (cur.x1[ch] - cur.x0[ch]) * kx;
                        J[1][ch] = (cur.y1[ch] - cur.y0[ch]) * ky;
                        J[2][ch] = (cur.z1[ch] - cur.z0[ch]) * kz;
                    }
                }
                const float x = irs_log_det_3x3(J);
                if (isfinite(x)) {
                    cnt[k] += 1.f;
                    const float dl = x - mu[k];
                    mu[k] += dl / cnt[k];
                    s2[k] += dl * (x - mu[k]);
                    if (mk[k]) {
                        s += (double)x;
                        sq += (double)x * (double)x;
                        ++n_fin;
                    }
                } else {
                    ++fo[k];
                    if (mk[k]) ++n_fold;
                }
            }
            cur = nxt;
            // this chain's mask sums over the warp (counts packed: at most 32 VW each), one slot per warp and chain of the chunk
            s = irs_warp_sum(s);
            sq = irs_warp_sum(sq);
            const unsigned packed = __reduce_add_sync(FULL, n_fold << 16 | n_fin);
            const int slot = c % CHUNK;
            if (lane == 0) { sh_s[slot][warp] = s; sh_q[slot][warp] = sq; sh_n[slot][warp] = packed; }
            if (slot == CHUNK - 1 || c == C - 1) {
                __syncthreads();
                const int c0 = c - slot;
                if ((int)threadIdx.x <= slot) {
                    const int t = threadIdx.x;
                    double a = 0.0, b = 0.0;
                    unsigned long long fin = 0ull, fold = 0ull;
                    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
                        a += sh_s[t][w];
                        b += sh_q[t][w];
                        fin += sh_n[t][w] & 0xffffu;
                        fold += sh_n[t][w] >> 16;
                    }
                    double* p = partials + (size_t)(c0 + t) * 2 * G + blockIdx.x;
                    p[0] = pass == 0 ? a : p[0] + a;
                    p[G] = pass == 0 ? b : p[G] + b;
                    if (fin | fold) atomicAdd(counters + c0 + t, fold << 32 | fin);
                    __threadfence();
                }
                __syncthreads();
            }
        }
        if (!active) continue;
        if constexpr (VW == 4) {
            *reinterpret_cast<int4*>(folds + i0) = make_int4(fo[0], fo[1], fo[2], fo[3]);
            *reinterpret_cast<float4*>(mean + i0) = make_float4(mu[0], mu[1], mu[2], mu[3]);
            *reinterpret_cast<float4*>(m2 + i0) = make_float4(s2[0], s2[1], s2[2], s2[3]);
        } else {
            folds[i0] = fo[0]; mean[i0] = mu[0]; m2[i0] = s2[0];
        }
    }
    // the last block to finish adds the partials of every block in index order: one warp per chain
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(counters + C, 1ull) == (unsigned long long)(G - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    for (int c = warp; c < C; c += blockDim.x >> 5) {
        const double* p = partials + (size_t)c * 2 * G;
        double a = 0.0, b = 0.0;
#pragma unroll 4
        for (int g = lane; g < G; g += 32) {
            a += __ldcg(p + g);
            b += __ldcg(p + G + g);
        }
        a = irs_warp_sum(a);
        b = irs_warp_sum(b);
        if (lane == 0) {
            const unsigned long long n = atomicExch(counters + c, 0ull);
            double* o = sample_stats + (size_t)c * 4;
            o[0] = (double)(n & 0xffffffffull);
            o[1] = (double)(n >> 32);
            o[2] = a;
            o[3] = b;
        }
    }
    if (threadIdx.x == 0) counters[C] = 0ull;
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// grid-stride over groups of VW voxels.  summary words: [0] sum folds, [1] voxels with folds > 0, [2] voxels with 2 folds > n,
// [3] voxels with n_v >= 1, [4] voxels with n_v >= 2, [7] voxels (all over the mask; integer atomics per block); [5], [6] the
// means of the mean and std maps (doubles, from partials [0, G) and [G, 2G) added in index order by the last block)
template <int VW>
__global__ void __launch_bounds__(256)
jacobian_posterior_kernel(const int* __restrict__ folds, const float* __restrict__ mean, const float* __restrict__ m2, int n,
                          long long V, const unsigned char* __restrict__ mask, float* __restrict__ p_fold,
                          float* __restrict__ mean_out, float* __restrict__ std_out, double* __restrict__ partials,
                          unsigned long long* __restrict__ counters, unsigned long long* __restrict__ summary) {
    __shared__ unsigned long long sh_i[6][8];
    __shared__ double sh_d[2][8];
    __shared__ bool last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, G = gridDim.x;
    const long long nq = V / VW;
    const float nf = (float)n;
    unsigned long long acc[6] = {0ull, 0ull, 0ull, 0ull, 0ull, 0ull};
    double sm = 0.0, ss = 0.0;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (long long)G * blockDim.x) {
        const long long i0 = q * VW;
        int fo[VW];
        float mu[VW], s2[VW], pf[VW], mo[VW], so[VW];
        unsigned char mk[VW];
        if constexpr (VW == 4) {
            const int4 f4 = __ldg(reinterpret_cast<const int4*>(folds + i0));
            const float4 a4 = __ldg(reinterpret_cast<const float4*>(mean + i0)), b4 = __ldg(reinterpret_cast<const float4*>(m2 + i0));
            const uchar4 m4 = *reinterpret_cast<const uchar4*>(mask + i0);
            fo[0] = f4.x; fo[1] = f4.y; fo[2] = f4.z; fo[3] = f4.w;
            mu[0] = a4.x; mu[1] = a4.y; mu[2] = a4.z; mu[3] = a4.w;
            s2[0] = b4.x; s2[1] = b4.y; s2[2] = b4.z; s2[3] = b4.w;
            mk[0] = m4.x; mk[1] = m4.y; mk[2] = m4.z; mk[3] = m4.w;
        } else {
            fo[0] = folds[i0]; mu[0] = mean[i0]; s2[0] = m2[i0]; mk[0] = mask[i0];
        }
#pragma unroll
        for (int k = 0; k < VW; ++k) {
            const int nv = n - fo[k];
            pf[k] = (float)fo[k] / nf;
            mo[k] = nv >= 1 ? mu[k] : NAN;
            so[k] = nv >= 2 ? sqrtf(s2[k] / (float)((double)nv - 1.0)) : NAN;   // welford_std_kernel's expression
            if (mk[k]) {
                acc[0] += (unsigned long long)fo[k];
                acc[1] += fo[k] > 0 ? 1ull : 0ull;
                acc[2] += 2ll * fo[k] > (long long)n ? 1ull : 0ull;
                acc[5] += 1ull;
                if (nv >= 1) { acc[3] += 1ull; sm += (double)mo[k]; }
                if (nv >= 2) { acc[4] += 1ull; ss += (double)so[k]; }
            }
        }
        if constexpr (VW == 4) {
            *reinterpret_cast<float4*>(p_fold + i0) = make_float4(pf[0], pf[1], pf[2], pf[3]);
            *reinterpret_cast<float4*>(mean_out + i0) = make_float4(mo[0], mo[1], mo[2], mo[3]);
            *reinterpret_cast<float4*>(std_out + i0) = make_float4(so[0], so[1], so[2], so[3]);
        } else {
            p_fold[i0] = pf[0]; mean_out[i0] = mo[0]; std_out[i0] = so[0];
        }
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[j] = warp_sum_u64(acc[j]);
    sm = irs_warp_sum(sm);
    ss = irs_warp_sum(ss);
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < 6; ++j) sh_i[j][warp] = acc[j];
        sh_d[0][warp] = sm;
        sh_d[1][warp] = ss;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nw = blockDim.x >> 5;
        for (int j = 0; j < 6; ++j) {
            unsigned long long t = 0ull;
            for (int w = 0; w < nw; ++w) t += sh_i[j][w];
            if (t) atomicAdd(summary + (j < 5 ? j : 7), t);
        }
        double a = 0.0, b = 0.0;
        for (int w = 0; w < nw; ++w) { a += sh_d[0][w]; b += sh_d[1][w]; }
        partials[blockIdx.x] = a;
        partials[G + blockIdx.x] = b;
        __threadfence();
        last = atomicAdd(counters, 1ull) == (unsigned long long)(G - 1);
    }
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    __threadfence();
    double a = 0.0, b = 0.0;
    for (int g = 0; g < G; ++g) {
        a += __ldcg(partials + g);
        b += __ldcg(partials + G + g);
    }
    const unsigned long long n1 = atomicAdd(summary + 3, 0ull), n2 = atomicAdd(summary + 4, 0ull);
    summary[5] = (unsigned long long)__double_as_longlong(n1 ? a / (double)n1 : (double)NAN);
    summary[6] = (unsigned long long)__double_as_longlong(n2 ? b / (double)n2 : (double)NAN);
    counters[0] = 0ull;
}

bool aligned(const void* p, unsigned bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0; }

unsigned reduce_grid(long long groups) {
    const long long b = (groups + 255) / 256;
    return (unsigned)(b < IRS_JACOBIAN_REDUCE_BLOCKS ? b : IRS_JACOBIAN_REDUCE_BLOCKS);
}

}  // namespace

extern "C" int irs_jacobian_update(const float* T, const unsigned char* mask, int C, int D, int H, int W, double count_before,
                                   int* folds, float* mean, float* m2, double* sample_stats, double* partials,
                                   unsigned long long* counters, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!T || !mask || !folds || !mean || !m2 || !sample_stats || !partials || !counters) return IRS_ERR_BAD_ARG;
    // the int32 folds and the fp32 running count are exact below 2^24 samples
    if (!(count_before >= 0.0) || count_before + C > 16777216.0) return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    IrsDims d{D, H, W};
    const bool vec = W % 4 == 0 && aligned(T, 16) && aligned(mask, 4) && aligned(folds, 16) && aligned(mean, 16) &&
                     aligned(m2, 16);
    if (vec)
        jacobian_update_kernel<4><<<reduce_grid(d.V() / 4), 256, 0, st>>>(T, mask, C, d, count_before, folds, mean, m2,
                                                                          partials, counters, sample_stats);
    else
        jacobian_update_kernel<1><<<reduce_grid(d.V()), 256, 0, st>>>(T, mask, C, d, count_before, folds, mean, m2,
                                                                      partials, counters, sample_stats);
    return (int)cudaGetLastError();
}

extern "C" int irs_jacobian_posterior(const int* folds, const float* mean, const float* m2, long long n, long long V,
                                      const unsigned char* mask, float* p_fold, float* mean_out, float* std_out,
                                      double* partials, unsigned long long* counters, long long* summary, void* stream) {
    if (!folds || !mean || !m2 || !mask || !p_fold || !mean_out || !std_out || !partials || !counters || !summary || n < 1 ||
        n > 16777216LL || V < 1 || V > 0x7fffffffLL)
        return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(summary, 0, sizeof(long long) * IRS_JACOBIAN_SUMMARY_WORDS, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(counters, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return (int)e;
    unsigned long long* sm = reinterpret_cast<unsigned long long*>(summary);
    const bool vec = V % 4 == 0 && aligned(folds, 16) && aligned(mean, 16) && aligned(m2, 16) && aligned(mask, 4) &&
                     aligned(p_fold, 16) && aligned(mean_out, 16) && aligned(std_out, 16);
    if (vec)
        jacobian_posterior_kernel<4><<<reduce_grid(V / 4), 256, 0, st>>>(folds, mean, m2, (int)n, V, mask, p_fold, mean_out,
                                                                         std_out, partials, counters, sm);
    else
        jacobian_posterior_kernel<1><<<reduce_grid(V), 256, 0, st>>>(folds, mean, m2, (int)n, V, mask, p_fold, mean_out,
                                                                     std_out, partials, counters, sm);
    return (int)cudaGetLastError();
}
