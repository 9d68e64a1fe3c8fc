// irs_smooth.cu -- Langevin proposal, Sobolev smoothing, diffusion regulariser, preconditioned SGD update
// (reference utils/functions.py:76-109, utils/util.py:48-58,394-404, utils/diff_op.py:78-96, model/loss.py:152-161,
//  trainer/trainer.py:351)
#include <mutex>

#include "irs_kernels.cuh"

namespace {

// out = v + coef * sigma * eps   (reference utils/util.py:48-58)
__global__ void __launch_bounds__(256)
langevin_kernel(const float* __restrict__ v, const float* __restrict__ sigma, long long sigma_cs, float coef,
                IrsRng rng, float* __restrict__ out, IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float* vc = v + (size_t)c * 3 * V;
    float* oc = out + (size_t)c * 3 * V;
    if (coef == 0.f) {
        oc[i] = vc[i]; oc[V + i] = vc[V + i]; oc[2 * V + i] = vc[2 * V + i];
        return;
    }
    float e[3];
    if (rng.explicit_values != nullptr) {
        const float* ec = rng.explicit_values + (size_t)c * 3 * V;
        e[0] = ec[i]; e[1] = ec[V + i]; e[2] = ec[2 * V + i];
    } else {
        const unsigned long long it = rng.iter_ptr ? (unsigned long long)(*rng.iter_ptr) : rng.iter;
        irs_normal3(rng.seed, (uint32_t)i, (uint32_t)(rng.chain0 + c), it, e);
    }
    float s0 = 1.f, s1 = 1.f, s2 = 1.f;
    if (sigma != nullptr) {
        const float* sc = sigma + (size_t)c * sigma_cs;
        s0 = sc[i]; s1 = sc[V + i]; s2 = sc[2 * V + i];
    }
    oc[i] = vc[i] + coef * s0 * e[0];
    oc[V + i] = vc[V + i] + coef * s1 * e[1];
    oc[2 * V + i] = vc[2 * V + i] + coef * s2 * e[2];
}

// one axis of the separable smoothing: out(j) = sum_t w_t in(clamp(j + t - s))  (replicate padding).  grid.y = C*3 fields.
// Interior voxels take a branch-free path with constant-stride loads; only the s voxels next to a face clamp indices.
template <int AXIS, int NT>
__global__ void __launch_bounds__(256)
smooth_axis_kernel(const float* __restrict__ in, float* __restrict__ out, IrsTaps taps, IrsDims d) {
    const int V = (int)d.V();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const float* f = in + (size_t)blockIdx.y * V;
    const int n = AXIS == 0 ? d.W : (AXIS == 1 ? d.H : d.D);
    const int stride = AXIS == 0 ? 1 : (AXIS == 1 ? d.W : d.W * d.H);
    const int j = AXIS == 0 ? i % d.W : (AXIS == 1 ? (i / d.W) % d.H : i / (d.W * d.H));
    constexpr int s = (NT - 1) / 2;
    float acc = 0.f;
    if (j >= s && j + s < n) {
        const float* p = f + (i - s * stride);
#pragma unroll
        for (int t = 0; t < NT; ++t) acc += taps.w[t] * __ldg(p + t * stride);
    } else {
        const int base = i - j * stride;
#pragma unroll
        for (int t = 0; t < NT; ++t) acc += taps.w[t] * __ldg(f + base + irs_clampi(j + t - s, 0, n - 1) * stride);
    }
    out[(size_t)blockIdx.y * V + i] = acc;
}

template <int NT>
static void launch_smooth3_nt(const float* in, float* work, float* out, const IrsTaps& taps, int C, IrsDims d,
                              cudaStream_t st) {
    dim3 grid((unsigned)((d.V() + 255) / 256), C * 3);
    smooth_axis_kernel<2, NT><<<grid, 256, 0, st>>>(in, out, taps, d);
    smooth_axis_kernel<1, NT><<<grid, 256, 0, st>>>(out, work, taps, d);
    smooth_axis_kernel<0, NT><<<grid, 256, 0, st>>>(work, out, taps, d);
}

// ---- 128-bit versions: one thread owns four consecutive x voxels (needs W % 4 == 0 and 16-byte aligned pointers) -----
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 fma4(float w, float4 a, float4 acc) {
    acc.x += w * a.x; acc.y += w * a.y; acc.z += w * a.z; acc.w += w * a.w;
    return acc;
}

template <int AXIS, int NT>   // AXIS 1 = y, 2 = z
__global__ void __launch_bounds__(256)
smooth_axis_vec_kernel(const float* __restrict__ in, float* __restrict__ out, IrsTaps taps, IrsDims d) {
    const int V = (int)d.V();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= V) return;
    const float* f = in + (size_t)blockIdx.y * V;
    const int n = AXIS == 1 ? d.H : d.D;
    const int stride = AXIS == 1 ? d.W : d.W * d.H;
    const int j = AXIS == 1 ? (i / d.W) % d.H : i / (d.W * d.H);
    constexpr int s = (NT - 1) / 2;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j >= s && j + s < n) {
        const float* p = f + (i - s * stride);
#pragma unroll
        for (int t = 0; t < NT; ++t) acc = fma4(taps.w[t], ld4(p + t * stride), acc);
    } else {
        const int base = i - j * stride;
#pragma unroll
        for (int t = 0; t < NT; ++t) acc = fma4(taps.w[t], ld4(f + base + irs_clampi(j + t - s, 0, n - 1) * stride), acc);
    }
    st4(out + (size_t)blockIdx.y * V + i, acc);
}

template <int NT>   // x axis: outputs x..x+3 need inputs x-s..x+3+s: three aligned float4 loads (s <= 4), clamped at row ends
__global__ void __launch_bounds__(256)
smooth_x_vec_kernel(const float* __restrict__ in, float* __restrict__ out, IrsTaps taps, IrsDims d) {
    const int V = (int)d.V();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= V) return;
    const float* f = in + (size_t)blockIdx.y * V;
    constexpr int s = (NT - 1) / 2;
    const int x = i % d.W;
    const float4 c = ld4(f + i);
    float w[12];
    const float4 l = x >= 4 ? ld4(f + i - 4) : make_float4(c.x, c.x, c.x, c.x);           // replicate the row's first value
    const float4 r = x + 4 < d.W ? ld4(f + i + 4) : make_float4(c.w, c.w, c.w, c.w);       // ... and its last value
    w[0] = l.x; w[1] = l.y; w[2] = l.z; w[3] = l.w; w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
    w[8] = r.x; w[9] = r.y; w[10] = r.z; w[11] = r.w;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int t = 0; t < NT; ++t) {
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] += taps.w[t] * w[4 + k + t - s];
    }
    st4(out + (size_t)blockIdx.y * V + i, make_float4(o[0], o[1], o[2], o[3]));
}

template <int NT>
static void launch_smooth3_vec_nt(const float* in, float* work, float* out, const IrsTaps& taps, int C, IrsDims d,
                                  cudaStream_t st) {
    dim3 grid((unsigned)((d.V() / 4 + 255) / 256), C * 3);
    smooth_axis_vec_kernel<2, NT><<<grid, 256, 0, st>>>(in, out, taps, d);
    smooth_axis_vec_kernel<1, NT><<<grid, 256, 0, st>>>(out, work, taps, d);
    smooth_x_vec_kernel<NT><<<grid, 256, 0, st>>>(work, out, taps, d);
}

static bool vec_ok(IrsDims d, const void* a, const void* b = nullptr, const void* c = nullptr, const void* e = nullptr) {
    auto al = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return d.W % 4 == 0 && al(a) && al(b) && al(c) && al(e);
}

__global__ void __launch_bounds__(256)
langevin_vec_kernel(const float* __restrict__ v, const float* __restrict__ sigma, long long sigma_cs, float coef,
                    IrsRng rng, float* __restrict__ out, IrsDims d) {
    const int V = (int)d.V();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float* vc = v + (size_t)c * 3 * V;
    float* oc = out + (size_t)c * 3 * V;
    float4 a[3] = {ld4(vc + i), ld4(vc + V + i), ld4(vc + 2 * V + i)};
    if (coef != 0.f) {
        float e[4][3];
        if (rng.explicit_values != nullptr) {
            const float* ec = rng.explicit_values + (size_t)c * 3 * V;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float4 t = ld4(ec + ch * V + i);
                e[0][ch] = t.x; e[1][ch] = t.y; e[2][ch] = t.z; e[3][ch] = t.w;
            }
        } else {
            const unsigned long long it = rng.iter_ptr ? (unsigned long long)(*rng.iter_ptr) : rng.iter;
#pragma unroll
            for (int k = 0; k < 4; ++k) irs_normal3(rng.seed, (uint32_t)(i + k), (uint32_t)(rng.chain0 + c), it, e[k]);
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            float4 sg = make_float4(1.f, 1.f, 1.f, 1.f);
            if (sigma != nullptr) sg = ld4(sigma + (size_t)c * sigma_cs + (size_t)ch * V + i);
            a[ch].x += coef * sg.x * e[0][ch]; a[ch].y += coef * sg.y * e[1][ch];
            a[ch].z += coef * sg.z * e[2][ch]; a[ch].w += coef * sg.w * e[3][ch];
        }
    }
    st4(oc + i, a[0]); st4(oc + V + i, a[1]); st4(oc + 2 * V + i, a[2]);
}

// ---- Langevin proposal + x and y smoothing in ONE kernel ---------------------------------------------------------------------
// A CTA owns TY full rows of one z-plane (all three components): the noisy state v + coef sigma eps of those rows plus a halo
// of s rows on either side goes to shared memory (the halo rows regenerate their Philox numbers -- a voxel's noise is a pure
// function of (seed, chain, iteration, voxel) -- 2 s / TY more generator work, against a whole pass over the field saved),
// is smoothed along x in place (one float4 per thread per round, neighbours read before anybody writes) and along y on the way
// out (a round of the in-place x pass takes whole rows, so that every unit reads neighbours no other round has written).  The
// z pass that follows is the only other pass: 12 + 12 (+ halo) read, 12 written here, 12 + 12 there, instead of four
// passes of 24 B.  Separable smoothing passes commute (replicate padding acts per axis), so x, y, z instead of the reference's
// z, y, x changes the result at rounding level only (checked against the oracle at 1e-5 like before).
template <int NT>
__global__ void __launch_bounds__(512, 2)
langevin_xy_kernel(const float* __restrict__ v, const float* __restrict__ sigma, long long sigma_cs, float coef, IrsRng rng,
                   float* __restrict__ out, IrsTaps taps, int TY, IrsDims d) {
    extern __shared__ __align__(16) float S[];   // [3][R][W], R = TY + 2 s
    constexpr int s = (NT - 1) / 2;
    const int V = (int)d.V(), W = d.W, W4 = W / 4, R = TY + 2 * s, CS = R * W;
    const int tiles_y = (d.H + TY - 1) / TY;
    const int z = blockIdx.x / tiles_y, y0 = (blockIdx.x - z * tiles_y) * TY;
    const int c = blockIdx.y;
    const float* vc = v + (size_t)c * 3 * V;
    const int units = R * W4;
    const unsigned long long it = (coef != 0.f && rng.explicit_values == nullptr)
                                      ? (rng.iter_ptr ? (unsigned long long)(*rng.iter_ptr) : rng.iter) : 0ull;
    // ---- noisy state of rows y0 - s .. y0 + TY - 1 + s (clamped = replicate padding along y) ----
    for (int u = threadIdx.x; u < units; u += blockDim.x) {
        const int r = u / W4, x4 = u - r * W4;
        const int gy = irs_clampi(y0 - s + r, 0, d.H - 1);
        const int i = (z * d.H + gy) * W + 4 * x4;
        float4 a[3] = {ld4(vc + i), ld4(vc + V + i), ld4(vc + 2 * V + i)};
        if (coef != 0.f) {
            float e[4][3];
            if (rng.explicit_values != nullptr) {
                const float* ec = rng.explicit_values + (size_t)c * 3 * V;
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    const float4 t = ld4(ec + ch * V + i);
                    e[0][ch] = t.x; e[1][ch] = t.y; e[2][ch] = t.z; e[3][ch] = t.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) irs_normal3(rng.seed, (uint32_t)(i + k), (uint32_t)(rng.chain0 + c), it, e[k]);
            }
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                float4 sg = make_float4(1.f, 1.f, 1.f, 1.f);
                if (sigma != nullptr) sg = ld4(sigma + (size_t)c * sigma_cs + (size_t)ch * V + i);
                a[ch].x += coef * sg.x * e[0][ch]; a[ch].y += coef * sg.y * e[1][ch];
                a[ch].z += coef * sg.z * e[2][ch]; a[ch].w += coef * sg.w * e[3][ch];
            }
        }
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) *reinterpret_cast<float4*>(S + ch * CS + r * W + 4 * x4) = a[ch];
    }
    __syncthreads();
    // ---- x pass, in place: every thread reads the three aligned float4 of its unit, then all write.  A round covers whole
    // rows (irs_langevin_fused keeps W4 <= 512), so no unit reads a neighbour that an earlier round already smoothed ----
    const int round_units = (blockDim.x / W4) * W4;
    for (int base = 0; base < units; base += round_units) {
        const int u = base + threadIdx.x;
        const bool valid = threadIdx.x < round_units && u < units;
        float4 o[3];
        if (valid) {
            const int r = u / W4, x4 = u - r * W4;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float* row = S + ch * CS + r * W;
                const float4 cc = *reinterpret_cast<const float4*>(row + 4 * x4);
                const float4 l = x4 > 0 ? *reinterpret_cast<const float4*>(row + 4 * x4 - 4) : make_float4(cc.x, cc.x, cc.x, cc.x);
                const float4 rr = x4 + 1 < W4 ? *reinterpret_cast<const float4*>(row + 4 * x4 + 4) : make_float4(cc.w, cc.w, cc.w, cc.w);
                const float w[12] = {l.x, l.y, l.z, l.w, cc.x, cc.y, cc.z, cc.w, rr.x, rr.y, rr.z, rr.w};
                float q[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int t = 0; t < NT; ++t) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) q[k] += taps.w[t] * w[4 + k + t - s];
                }
                o[ch] = make_float4(q[0], q[1], q[2], q[3]);
            }
        }
        __syncthreads();
        if (valid) {
            const int r = u / W4, x4 = u - r * W4;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) *reinterpret_cast<float4*>(S + ch * CS + r * W + 4 * x4) = o[ch];
        }
        __syncthreads();
    }
    // ---- y pass on the way out ----
    float* oc = out + (size_t)c * 3 * V;
    for (int u = threadIdx.x; u < TY * W4; u += blockDim.x) {
        const int ry = u / W4, x4 = u - ry * W4, y = y0 + ry;
        if (y >= d.H) continue;
        const int i = (z * d.H + y) * W + 4 * x4;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* col = S + ch * CS + ry * W + 4 * x4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int t = 0; t < NT; ++t) acc = fma4(taps.w[t], *reinterpret_cast<const float4*>(col + t * W), acc);
            st4(oc + ch * V + i, acc);
        }
    }
}

template <int NT>
static int launch_langevin_xy_nt(const float* v, const float* sigma, long long sigma_cs, float coef, const IrsRng& rng,
                                 float* work, float* out, const IrsTaps& taps, int C, IrsDims d, cudaStream_t st) {
    constexpr int s = (NT - 1) / 2;
    int TY = 32;
    while (TY > 8 && (size_t)3 * (TY + 2 * s) * d.W * 4 > 100 * 1024) TY -= 8;
    if (TY > d.H) TY = d.H;
    const size_t smem = (size_t)3 * (TY + 2 * s) * d.W * 4;
    if (smem > 200 * 1024) return IRS_ERR_UNSUPPORTED;
    static std::mutex mu;
    static bool ready[64] = {};
    {
        std::lock_guard<std::mutex> lock(mu);
        int dev = 0;
        cudaGetDevice(&dev);
        if (!ready[dev & 63]) {
            cudaError_t e = cudaFuncSetAttribute(langevin_xy_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (e != cudaSuccess) return (int)e;
            ready[dev & 63] = true;
        }
    }
    dim3 grid((unsigned)(((d.H + TY - 1) / TY) * d.D), C);
    langevin_xy_kernel<NT><<<grid, 512, smem, st>>>(v, sigma, sigma_cs, coef, rng, work, taps, TY, d);
    dim3 vgrid((unsigned)((d.V() / 4 + 255) / 256), C * 3);
    smooth_axis_vec_kernel<2, NT><<<vgrid, 256, 0, st>>>(work, out, taps, d);
    return (int)cudaGetLastError();
}

// d energy / d v for four consecutive x voxels of one channel (row neighbours from the aligned neighbours l, r)
__device__ __forceinline__ float4 energy_grad4(const float* __restrict__ f, int i, int x, int y, int z, IrsDims d) {
    const int sy = d.W, sz = d.W * d.H;
    const float4 c = ld4(f + i);
    // interior (no voxel of the four touches a face or the doubled last difference): the same operations as
    // irs_diff_energy_grad with all weights one, without its six position tests per voxel and axis
    if (x >= 4 && x + 8 <= d.W && y >= 1 && y + 3 <= d.H && z >= 1 && z + 3 <= d.D) {
        const float lft = __ldg(f + i - 1), rgt = __ldg(f + i + 4);
        const float4 ym = ld4(f + i - sy), yp = ld4(f + i + sy), zm = ld4(f + i - sz), zp = ld4(f + i + sz);
        auto g1 = [](float vm, float vj, float vp) { return 2.0f * ((vj - vm) - (vp - vj)); };
        float4 g;
        g.x = g1(lft, c.x, c.y) + g1(ym.x, c.x, yp.x) + g1(zm.x, c.x, zp.x);
        g.y = g1(c.x, c.y, c.z) + g1(ym.y, c.y, yp.y) + g1(zm.y, c.y, zp.y);
        g.z = g1(c.y, c.z, c.w) + g1(ym.z, c.z, yp.z) + g1(zm.z, c.z, zp.z);
        g.w = g1(c.z, c.w, rgt) + g1(ym.w, c.w, yp.w) + g1(zm.w, c.w, zp.w);
        return g;
    }
    const float lft = x > 0 ? __ldg(f + i - 1) : 0.f, rgt = x + 4 < d.W ? __ldg(f + i + 4) : 0.f;
    const float4 ym = y > 0 ? ld4(f + i - sy) : c, yp = y < d.H - 1 ? ld4(f + i + sy) : c;
    const float4 zm = z > 0 ? ld4(f + i - sz) : c, zp = z < d.D - 1 ? ld4(f + i + sz) : c;
    float4 g;
    g.x = irs_diff_energy_grad(lft, c.x, c.y, x, d.W) + irs_diff_energy_grad(ym.x, c.x, yp.x, y, d.H) + irs_diff_energy_grad(zm.x, c.x, zp.x, z, d.D);
    g.y = irs_diff_energy_grad(c.x, c.y, c.z, x + 1, d.W) + irs_diff_energy_grad(ym.y, c.y, yp.y, y, d.H) + irs_diff_energy_grad(zm.y, c.y, zp.y, z, d.D);
    g.z = irs_diff_energy_grad(c.y, c.z, c.w, x + 2, d.W) + irs_diff_energy_grad(ym.z, c.z, yp.z, y, d.H) + irs_diff_energy_grad(zm.z, c.z, zp.z, z, d.D);
    g.w = irs_diff_energy_grad(c.z, c.w, rgt, x + 3, d.W) + irs_diff_energy_grad(ym.w, c.w, yp.w, y, d.H) + irs_diff_energy_grad(zm.w, c.w, zp.w, z, d.D);
    return g;
}

__global__ void __launch_bounds__(256)
sgd_update_vec_kernel(float* __restrict__ v, const float* __restrict__ sigma, long long sigma_cs,
                      const float* __restrict__ css, const float* __restrict__ g_css, const double* __restrict__ coef,
                      long long coef_stride, float tau, float* __restrict__ grad_v, IrsDims d) {
    const int V = (int)d.V();
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float k = (float)coef[(size_t)c * coef_stride];
    const int x = i % d.W, y = (i / d.W) % d.H, z = i / (d.W * d.H);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const size_t o = ((size_t)c * 3 + ch) * V + i;
        const float4 ge = energy_grad4(css + ((size_t)c * 3 + ch) * V, i, x, y, z, d);
        const float4 gc = ld4(g_css + o);
        float4 sg = make_float4(1.f, 1.f, 1.f, 1.f);
        if (sigma != nullptr) sg = ld4(sigma + (size_t)c * sigma_cs + (size_t)ch * V + i);
        float4 g, vv = *reinterpret_cast<const float4*>(v + o);
        g.x = sg.x * sg.x * (gc.x + k * ge.x); g.y = sg.y * sg.y * (gc.y + k * ge.y);
        g.z = sg.z * sg.z * (gc.z + k * ge.z); g.w = sg.w * sg.w * (gc.w + k * ge.w);
        if (grad_v != nullptr) st4(grad_v + o, g);
        vv.x -= tau * g.x; vv.y -= tau * g.y; vv.z -= tau * g.z; vv.w -= tau * g.w;
        st4(v + o, vv);
    }
}

__global__ void __launch_bounds__(256)
reg_energy_vec_kernel(const float* __restrict__ v, double* __restrict__ energy, long long energy_stride,
                      double* __restrict__ partials, unsigned int* __restrict__ counters, IrsDims d) {
    __shared__ double sh[32];
    __shared__ double total[1];
    const int V = (int)d.V(), sy = d.W, sz = d.W * d.H;
    const int c = blockIdx.y;
    const float* vc = v + (size_t)c * 3 * V;
    float acc = 0.f;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4; i < V; i += gridDim.x * blockDim.x * 4) {
        const int x = i % d.W, y = (i / d.W) % d.H, z = i / sz;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* f = vc + (size_t)ch * V;
            const float4 a = ld4(f + i);
            const float nx = x + 4 < d.W ? __ldg(f + i + 4) : 0.f;
            const float4 py = y < d.H - 1 ? ld4(f + i + sy) : a, pz = z < d.D - 1 ? ld4(f + i + sz) : a;
            acc += irs_diff_energy(a.x, a.y, x, d.W) + irs_diff_energy(a.y, a.z, x + 1, d.W) +
                   irs_diff_energy(a.z, a.w, x + 2, d.W) + irs_diff_energy(a.w, nx, x + 3, d.W);
            acc += irs_diff_energy(a.x, py.x, y, d.H) + irs_diff_energy(a.y, py.y, y, d.H) +
                   irs_diff_energy(a.z, py.z, y, d.H) + irs_diff_energy(a.w, py.w, y, d.H);
            acc += irs_diff_energy(a.x, pz.x, z, d.D) + irs_diff_energy(a.y, pz.y, z, d.D) +
                   irs_diff_energy(a.z, pz.z, z, d.D) + irs_diff_energy(a.w, pz.w, z, d.D);
        }
    }
    double blk[1];
    irs_block_sum<1>(&acc, blk, sh);
    if (irs_grid_sum<1>(blk, partials + (size_t)c * gridDim.x, counters + c, total)) {
        if (threadIdx.x == 0) energy[(size_t)c * energy_stride] = total[0];
    }
}

// energy of one chain: sum over 3 components x 3 axes of squared forward differences (last one counted twice)
__global__ void __launch_bounds__(256)
reg_energy_kernel(const float* __restrict__ v, double* __restrict__ energy, long long energy_stride,
                  double* __restrict__ partials, unsigned int* __restrict__ counters, IrsDims d) {
    __shared__ double sh[32];
    __shared__ double total[1];
    const long long V = d.V();
    const int c = blockIdx.y;
    const float* vc = v + (size_t)c * 3 * V;
    float acc = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
        const long long sy = d.W, sz = (long long)d.W * d.H;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const float* f = vc + (size_t)ch * V;
            const float vj = f[i];
            const float vx = x < d.W - 1 ? __ldg(f + i + 1) : 0.f;
            const float vy = y < d.H - 1 ? __ldg(f + i + sy) : 0.f;
            const float vz = z < d.D - 1 ? __ldg(f + i + sz) : 0.f;
            acc += irs_diff_energy(vj, vx, x, d.W) + irs_diff_energy(vj, vy, y, d.H) + irs_diff_energy(vj, vz, z, d.D);
        }
    }
    double blk[1];
    irs_block_sum<1>(&acc, blk, sh);
    if (irs_grid_sum<1>(blk, partials + (size_t)c * gridDim.x, counters + c, total)) {
        if (threadIdx.x == 0) energy[(size_t)c * energy_stride] = total[0];
    }
}

__global__ void __launch_bounds__(256)
reg_energy_grad_kernel(const float* __restrict__ v, const double* __restrict__ coef, float* __restrict__ g_v,
                       IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float k = (float)coef[c];
    const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
    const long long sy = d.W, sz = (long long)d.W * d.H;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const float* f = v + ((size_t)c * 3 + ch) * V;
        const float vj = f[i];
        float ge = irs_diff_energy_grad(x > 0 ? __ldg(f + i - 1) : 0.f, vj, x < d.W - 1 ? __ldg(f + i + 1) : 0.f, x, d.W)
                 + irs_diff_energy_grad(y > 0 ? __ldg(f + i - sy) : 0.f, vj, y < d.H - 1 ? __ldg(f + i + sy) : 0.f, y, d.H)
                 + irs_diff_energy_grad(z > 0 ? __ldg(f + i - sz) : 0.f, vj, z < d.D - 1 ? __ldg(f + i + sz) : 0.f, z, d.D);
        g_v[((size_t)c * 3 + ch) * V + i] += k * ge;
    }
}

// grad_v = sigma^2 (g_css + coef_c dE/dcss) ;  v <- v - tau grad_v    (reference utils/functions.py:82-84 + plain SGD)
__global__ void __launch_bounds__(256)
sgd_update_kernel(float* __restrict__ v, const float* __restrict__ sigma, long long sigma_cs,
                  const float* __restrict__ css, const float* __restrict__ g_css, const double* __restrict__ coef,
                  long long coef_stride, float tau, float* __restrict__ grad_v, IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float k = (float)coef[(size_t)c * coef_stride];
    const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
    const long long sy = d.W, sz = (long long)d.W * d.H;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const size_t o = ((size_t)c * 3 + ch) * V + i;
        const float* f = css + ((size_t)c * 3 + ch) * V;
        const float vj = f[i];
        float ge = irs_diff_energy_grad(x > 0 ? __ldg(f + i - 1) : 0.f, vj, x < d.W - 1 ? __ldg(f + i + 1) : 0.f, x, d.W)
                 + irs_diff_energy_grad(y > 0 ? __ldg(f + i - sy) : 0.f, vj, y < d.H - 1 ? __ldg(f + i + sy) : 0.f, y, d.H)
                 + irs_diff_energy_grad(z > 0 ? __ldg(f + i - sz) : 0.f, vj, z < d.D - 1 ? __ldg(f + i + sz) : 0.f, z, d.D);
        const float sg = sigma ? sigma[(size_t)c * sigma_cs + (size_t)ch * V + i] : 1.f;
        const float g = sg * sg * (g_css[o] + k * ge);
        if (grad_v != nullptr) grad_v[o] = g;
        v[o] -= tau * g;
    }
}

// nabla (C,3,D,H,W,3): [c, j, voxel, i] = d v_i / d x_j   (reference utils/diff_op.py:78-96)
__global__ void __launch_bounds__(256)
diff_fwd_kernel(const float* __restrict__ v, float* __restrict__ nabla, int transformation, IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
    const long long sy = d.W, sz = (long long)d.W * d.H;
    // replicated last difference: position n-1 repeats the difference of position n-2
    const long long ix = x < d.W - 1 ? i : i - 1, iy = y < d.H - 1 ? i : i - sy, iz = z < d.D - 1 ? i : i - sz;
    float sxp = 1.f, syp = 1.f, szp = 1.f;
    if (transformation) {
        sxp = (float)(d.W - 1) * 0.5f; syp = (float)(d.H - 1) * 0.5f; szp = (float)(d.D - 1) * 0.5f;
    }
    float* o = nabla + (size_t)c * 9 * V;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        const float* f = v + ((size_t)c * 3 + ch) * V;
        o[(0 * V + i) * 3 + ch] = (__ldg(f + ix + 1) - __ldg(f + ix)) * sxp;
        o[(1 * V + i) * 3 + ch] = (__ldg(f + iy + sy) - __ldg(f + iy)) * syp;
        o[(2 * V + i) * 3 + ch] = (__ldg(f + iz + sz) - __ldg(f + iz)) * szp;
    }
}

// adjoint of diff_fwd: g_v[ch](j) = sum over axes of  [G(j-1) - G(j)] with the replicated last entry folded back
__global__ void __launch_bounds__(256)
diff_bwd_kernel(const float* __restrict__ g_nabla, float* __restrict__ g_v, int transformation, IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
    const long long st[3] = {1, d.W, (long long)d.W * d.H};
    const int pos[3] = {x, y, z}, len[3] = {d.W, d.H, d.D};
    const float* G = g_nabla + (size_t)c * 9 * V;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        float acc = 0.f;
#pragma unroll
        for (int ax = 0; ax < 3; ++ax) {
            const int j = pos[ax], n = len[ax];
            const float sp = transformation ? (float)(n - 1) * 0.5f : 1.f;
            const float* Ga = G + (size_t)ax * V * 3;
            // effective gradient on difference d_m (m = 0..n-2): Ge(m) = G(m) + [m == n-2] G(n-1)
            float a = 0.f;
            if (j >= 1) {  // + Ge(j-1)
                const int m = j - 1;
                float ge = __ldg(Ga + (i - st[ax]) * 3 + ch);
                if (m == n - 2) ge += __ldg(Ga + i * 3 + ch);  // here i is position n-1
                a += ge;
            }
            if (j <= n - 2) {  // - Ge(j)
                float ge = __ldg(Ga + i * 3 + ch);
                if (j == n - 2) ge += __ldg(Ga + (i + st[ax]) * 3 + ch);
                a -= ge;
            }
            acc += a * sp;
        }
        g_v[((size_t)c * 3 + ch) * V + i] = acc;
    }
}

}  // namespace

int irs_launch_langevin(const float* v, const float* sigma, long long sigma_cs, float coef, IrsRng rng, float* out,
                        int C, IrsDims d, cudaStream_t st) {
    if (vec_ok(d, v, sigma, out, rng.explicit_values) && (sigma_cs % 4) == 0) {
        dim3 vgrid((unsigned)((d.V() / 4 + 255) / 256), C);
        langevin_vec_kernel<<<vgrid, 256, 0, st>>>(v, sigma, sigma_cs, coef, rng, out, d);
        return (int)cudaGetLastError();
    }
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    langevin_kernel<<<grid, 256, 0, st>>>(v, sigma, sigma_cs, coef, rng, out, d);
    return (int)cudaGetLastError();
}

// in -> (z pass) out -> (y pass) work -> (x pass) out : the reference's order (utils/util.py:402-404)
int irs_launch_smooth3(const float* in, float* work, float* out, const IrsTaps& taps, int C, IrsDims d,
                       cudaStream_t st) {
    if (vec_ok(d, in, work, out) && taps.n <= 9) {
        switch (taps.n) {
            case 3: launch_smooth3_vec_nt<3>(in, work, out, taps, C, d, st); break;
            case 5: launch_smooth3_vec_nt<5>(in, work, out, taps, C, d, st); break;
            case 7: launch_smooth3_vec_nt<7>(in, work, out, taps, C, d, st); break;
            case 9: launch_smooth3_vec_nt<9>(in, work, out, taps, C, d, st); break;
            default: return IRS_ERR_UNSUPPORTED;
        }
        return (int)cudaGetLastError();
    }
    switch (taps.n) {
        case 3: launch_smooth3_nt<3>(in, work, out, taps, C, d, st); break;
        case 5: launch_smooth3_nt<5>(in, work, out, taps, C, d, st); break;
        case 7: launch_smooth3_nt<7>(in, work, out, taps, C, d, st); break;
        case 9: launch_smooth3_nt<9>(in, work, out, taps, C, d, st); break;
        case 11: launch_smooth3_nt<11>(in, work, out, taps, C, d, st); break;
        case 13: launch_smooth3_nt<13>(in, work, out, taps, C, d, st); break;
        case 15: launch_smooth3_nt<15>(in, work, out, taps, C, d, st); break;
        default: return IRS_ERR_UNSUPPORTED;
    }
    return (int)cudaGetLastError();
}

// the smallest tile (8 rows + halo) fits in 200 KB, and a round of the x pass (512 threads, one float4 each) holds at least
// one whole row (implied by the first condition today: W <= 1706; stated so that a larger tile budget cannot make it spin)
bool irs_langevin_fused(IrsDims d, int n_taps) {
    return d.W % 4 == 0 && (n_taps == 3 || n_taps == 5 || n_taps == 7) && (size_t)3 * (8 + n_taps - 1) * d.W * 4 <= 200 * 1024 &&
           d.W / 4 <= 512;
}

// Langevin proposal + separable smoothing: two kernels (noise + x + y on shared-memory rows, then z) when the field can be
// vectorised, the four-pass sequence otherwise.
int irs_launch_langevin_smooth3(const float* v, const float* sigma, long long sigma_cs, float coef, IrsRng rng, float* work,
                                float* out, const IrsTaps& taps, int C, IrsDims d, cudaStream_t st) {
    if (irs_langevin_fused(d, taps.n) && vec_ok(d, v, sigma, out, rng.explicit_values) && vec_ok(d, work) &&
        (sigma_cs % 4) == 0) {
        switch (taps.n) {
            case 3: return launch_langevin_xy_nt<3>(v, sigma, sigma_cs, coef, rng, work, out, taps, C, d, st);
            case 5: return launch_langevin_xy_nt<5>(v, sigma, sigma_cs, coef, rng, work, out, taps, C, d, st);
            default: return launch_langevin_xy_nt<7>(v, sigma, sigma_cs, coef, rng, work, out, taps, C, d, st);
        }
    }
    IRS_TRY(irs_launch_langevin(v, sigma, sigma_cs, coef, rng, work, C, d, st));
    return irs_launch_smooth3(work, work, out, taps, C, d, st);
}

int irs_reg_energy_blocks(IrsDims d) {
    long long b = (d.V() + 255) / 256;
    return (int)(b < 592 ? b : 592);  // 4 CTAs per SM x 148 SMs
}

int irs_launch_reg_energy(const float* v, double* energy, long long energy_stride, double* partials,
                          unsigned int* counters, int C, IrsDims d, cudaStream_t st) {
    dim3 grid(irs_reg_energy_blocks(d), C);
    if (vec_ok(d, v)) reg_energy_vec_kernel<<<grid, 256, 0, st>>>(v, energy, energy_stride, partials, counters, d);
    else reg_energy_kernel<<<grid, 256, 0, st>>>(v, energy, energy_stride, partials, counters, d);
    return (int)cudaGetLastError();
}

int irs_launch_sgd_update(float* v, const float* sigma, long long sigma_cs, const float* css, const float* g_css,
                          const double* coef, long long coef_stride, float tau, float* grad_v, int C, IrsDims d,
                          cudaStream_t st) {
    if (vec_ok(d, v, sigma, css, g_css) && vec_ok(d, grad_v) && (sigma_cs % 4) == 0) {
        dim3 vgrid((unsigned)((d.V() / 4 + 255) / 256), C);
        sgd_update_vec_kernel<<<vgrid, 256, 0, st>>>(v, sigma, sigma_cs, css, g_css, coef, coef_stride, tau, grad_v, d);
        return (int)cudaGetLastError();
    }
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    sgd_update_kernel<<<grid, 256, 0, st>>>(v, sigma, sigma_cs, css, g_css, coef, coef_stride, tau, grad_v, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_langevin_sobolev(const float* v, const float* sigma, long long sigma_cs, float coef,
                                    const float* eps, unsigned long long seed, unsigned long long iter, int chain0,
                                    const float* taps_host, int n_taps, float* work, float* out, int C, int D, int H,
                                    int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!v || !out) return IRS_ERR_BAD_ARG;
    if (n_taps < 0 || n_taps > IRS_MAX_TAPS || (n_taps > 0 && (n_taps % 2 == 0 || !taps_host || !work)))
        return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    cudaStream_t st = (cudaStream_t)stream;
    IrsRng rng{eps, seed, nullptr, iter, chain0};
    if (n_taps == 0) return irs_launch_langevin(v, sigma, sigma_cs, coef, rng, out, C, d, st);
    IrsTaps taps;
    taps.n = n_taps;
    for (int t = 0; t < n_taps; ++t) taps.w[t] = taps_host[t];
    return irs_launch_langevin_smooth3(v, sigma, sigma_cs, coef, rng, work, out, taps, C, d, st);
}

extern "C" int irs_diff_fwd(const float* v, float* nabla, int transformation, int C, int D, int H, int W,
                            void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!v || !nabla) return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    diff_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(v, nabla, transformation, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_diff_bwd(const float* g_nabla, float* g_v, int transformation, int C, int D, int H, int W,
                            void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!g_nabla || !g_v) return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    diff_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g_nabla, g_v, transformation, d);
    return (int)cudaGetLastError();
}

extern "C" size_t irs_reduce_scratch_doubles(int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    return (size_t)C * 592 * 32;
}

extern "C" int irs_reg_energy(const float* v, double* energy, double* partials, unsigned int* counters, int C, int D,
                              int H, int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!v || !energy || !partials || !counters) return IRS_ERR_BAD_ARG;
    return irs_launch_reg_energy(v, energy, 1, partials, counters, C, IrsDims{D, H, W}, (cudaStream_t)stream);
}

extern "C" int irs_reg_energy_grad(const float* v, const double* coef, float* g_v, int C, int D, int H, int W,
                                   void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!v || !coef || !g_v) return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    reg_energy_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(v, coef, g_v, d);
    return (int)cudaGetLastError();
}
