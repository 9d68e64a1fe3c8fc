// irs_svf.cu -- scaling and squaring of a stationary velocity field and its adjoint
// (reference utils/transformation.py:63-76 = 12 x F.grid_sample; backward = 12 x grid_sampler_3d_backward)
//
// Voxel-unit recurrence (SURVEY Appendix A.6):
//   u_0 = v / 2^n ;  u_{k+1}(i) = u_k(i) + trilinear[u_k]( clamp(i + u_k(i)) )
// Adjoint of one step, g' = dL/du_{k+1}:
//   g(t) = g'(t)                                              direct
//        + inside(t) * sum_c g'_c(t) * grad trilinear[u_c](p(t))   position term (gather)
//        + sum_s  w(p(s) - t) * g'(s)                         interpolation transpose
// The transpose is evaluated as a GATHER over the sources s in a window of radius R = floor(max|u_k|) + 1 around t
// (every s with a non-zero hat weight lies inside it), so no atomics are issued -- ATen scatters 24 atomicAdds per
// voxel here.  Candidates are pruned axis by axis (a zero x-weight skips the y/z loads).  For R above
// gather_radius_max the exact scatter kernel below takes over (large deformations; still CUDA, no CPU path).
//
// Kernels in this file, fastest first; the choice between them is made on the device from max|u_k| (no host sync):
//   svf_step_fwd_tma_kernel    forward step, TMA plane ring (max|u| < 1 bound; otherwise its in-kernel ring fallback)
//   svf_step_bwd_tma2_kernel   adjoint step, TMA rings + per-source records, two targets per thread
//   svf_step_fwd_tile_kernel / svf_step_bwd_tile_kernel   shared-memory rings fed by ordinary loads: row pitches the TMA
//                              unit cannot address (W % 4 != 0), and steps with 1 <= max|u| < 2 inside the TMA kernels
//   irs_body_svf_fwd / irs_body_svf_bwd, svf_step_bwd_scatter_kernel   global gathers / atomic scatter for larger radii
#include <cstdlib>
#include <mutex>

#include "irs_kernels.cuh"
#include "irs_bodies.cuh"
#include "irs_tma.cuh"

namespace {

__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {
    atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

// ---------------------------------------------------------------------------------------------------------------------
// Cell map: besides the global max |u_k| of a step, the forward pass leaves (for steps that reach one voxel) the maximum
// over cells of 32 x 8 x 8 voxels.  The adjoint of a tile then depends on the displacements NEAR that tile only: a tile
// whose neighbourhood stays below one voxel takes the TMA kernel even when the field exceeds one voxel elsewhere (typical
// for a registration: large deformations are local).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int CELL_X = 32, CELL_Y = 8, CELL_Z = 8;
struct IrsCells {
    float* p;          // this step's map, (C, nz, ny, nx) floats, or nullptr
    int nx, ny, nz;
};
__host__ __device__ inline int irs_cells_per_chain(IrsDims d) {
    return ((d.W + CELL_X - 1) / CELL_X) * ((d.H + CELL_Y - 1) / CELL_Y) * ((d.D + CELL_Z - 1) / CELL_Z);
}
static IrsCells make_cells(float* maxabs, int n_steps, int k, int C, IrsDims d) {
    IrsCells c;
    c.nx = (d.W + CELL_X - 1) / CELL_X; c.ny = (d.H + CELL_Y - 1) / CELL_Y; c.nz = (d.D + CELL_Z - 1) / CELL_Z;
    c.p = maxabs + n_steps + (size_t)k * C * c.nx * c.ny * c.nz;
    return c;
}
// maximum of the cell map over the cells that overlap the voxel box [x0,x1] x [y0,y1] x [z0,z1]; all threads get it
__device__ __forceinline__ float cells_region_max(const IrsCells& cm, int chain, int x0, int x1, int y0, int y1, int z0,
                                                  int z1) {
    __shared__ float s_region_max;
    const int cx0 = max(x0, 0) / CELL_X, cx1 = min(x1 / CELL_X, cm.nx - 1), cy0 = max(y0, 0) / CELL_Y,
              cy1 = min(y1 / CELL_Y, cm.ny - 1), cz0 = max(z0, 0) / CELL_Z, cz1 = min(z1 / CELL_Z, cm.nz - 1);
    if (threadIdx.x < 32) {
        const int nx = cx1 - cx0 + 1, ny = cy1 - cy0 + 1, nz = cz1 - cz0 + 1, n = nx * ny * nz;
        float m = 0.f;
        for (int i = threadIdx.x; i < n; i += 32) {
            const int ix = i % nx, iy = (i / nx) % ny, iz = i / (nx * ny);
            m = fmaxf(m, __ldg(cm.p + (((size_t)chain * cm.nz + cz0 + iz) * cm.ny + cy0 + iy) * cm.nx + cx0 + ix));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (threadIdx.x == 0) s_region_max = m;
    }
    __syncthreads();
    const float r = s_region_max;
    __syncthreads();
    return r;
}

// Cell map of one field, computed only when somebody needs it: the step's max |u| has reached one voxel (the adjoint then
// picks its window per tile).  One block per cell; launched behind the last forward steps, exits at once otherwise.
// blockIdx.z selects the step k = k_first + z: ONE launch behind the forward pass covers the (up to four) late steps that can
// reach one voxel -- as four launches the early exits alone cost ~2.5 us each in every transition.
__global__ void __launch_bounds__(256)
svf_cells_kernel(const float* __restrict__ v_all, const float* __restrict__ hist, float scale0, float* __restrict__ maxabs,
                 int n_steps, int k_first, long long F, int C, IrsDims d) {
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    const int k = k_first + blockIdx.z;
    if ((int)floorf(__ldg(maxabs + k) + 1e-3f) + 1 < 2) return;   // = svf_gather_radius(max |u_k|) < 2: nobody reads the map
    IrsCells cm;
    cm.nx = (d.W + CELL_X - 1) / CELL_X; cm.ny = (d.H + CELL_Y - 1) / CELL_Y; cm.nz = (d.D + CELL_Z - 1) / CELL_Z;
    cm.p = maxabs + n_steps + (size_t)k * C * cm.nx * cm.ny * cm.nz;
    const float* u_all = (k == 0) ? v_all : hist + (size_t)(k - 1) * F;
    const float scale = (k == 0) ? scale0 : 1.0f;
    const int cx = blockIdx.x % cm.nx, cy = (blockIdx.x / cm.nx) % cm.ny, cz = blockIdx.x / (cm.nx * cm.ny), chain = blockIdx.y;
    const int V = (int)d.V();
    const float* u = u_all + (size_t)chain * 3 * V;
    const int lx = threadIdx.x % CELL_X, ly = threadIdx.x / CELL_X;   // 32 x 8 threads = one plane of the cell
    const int x = cx * CELL_X + lx, y = cy * CELL_Y + ly;
    float m = 0.f;
    if (x < d.W && y < d.H) {
        for (int z = cz * CELL_Z; z < min((cz + 1) * CELL_Z, d.D); ++z) {
            const int i = (z * d.H + y) * d.W + x;
            m = fmaxf(m, fmaxf(fabsf(__ldg(u + i)), fmaxf(fabsf(__ldg(u + V + i)), fabsf(__ldg(u + 2 * V + i)))));
        }
    }
    m *= scale;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float mm = sm[0];
        for (int w = 1; w < 8; ++w) mm = fmaxf(mm, sm[w]);
        cm.p[(((size_t)chain * cm.nz + cz) * cm.ny + cy) * cm.nx + cx] = mm;
    }
}

// exact scatter form of the interpolation transpose for steps whose displacement exceeds the gather window.
// Launched after every tiled adjoint step with a small persistent grid: when the step was handled by the gather
// (the normal case) all CTAs leave after one uniform load -- a full-size grid of empty CTAs would cost ~7 us per step.
__global__ void __launch_bounds__(256)
svf_step_bwd_scatter_kernel(const float* __restrict__ in, float in_scale, const float* __restrict__ gp_all,
                            float* __restrict__ g_all, const float* __restrict__ maxabs, int radius_max,
                            float out_scale, int C, IrsDims d) {
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    const int R = (int)floorf(__ldg(maxabs) + 1e-3f) + 1;   // = svf_gather_radius
    if (R <= radius_max) return;
    const long long V = d.V();
    for (int c = 0; c < C; ++c) {
        const size_t off = (size_t)c * 3 * V;
        float* g = g_all + off;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x)
            irs_body_svf_bwd_scatter(in + off, in_scale, gp_all + off, out_scale, V, i, d,
                                     [&](long long t, int ch, float val) { atomicAdd(g + (size_t)ch * V + t, val); });
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Tiled kernels.  A CTA owns a TX x TY column of voxels and marches along z.  The velocity planes z-R..z+R live in a
// shared-memory ring (halo R in x and y, zero outside the volume), so every trilinear corner and every candidate
// source of the interpolation transpose is a shared-memory load with a compile-time offset.  The next plane is
// prefetched into registers while the current one is processed.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TILE_X = 32, TILE_Y = 8, TILE_T = TILE_X * TILE_Y;

// EX = valid row width, RS = row stride in shared memory.  RS is a multiple of 32 floats so that all rows alias the same
// banks: the lanes of a warp sit in distinct columns, hence gathers whose cells lie in different rows do not conflict
// (with RS = EX = 36 a lane pair 4 apart in neighbouring rows collides -- measured 2.4 wavefronts per load).
// The forward kernel (R = 2, data-dependent cells) pads; the adjoint's R = 1 path reads candidates at fixed offsets
// from the thread's own column (conflict-free with RS = EX) and prefers the smaller footprint.
template <int R, bool PAD = false>
struct Tile {
    static constexpr int EX = TILE_X + 2 * R, EY = TILE_Y + 2 * R, RS = PAD ? 64 : EX, PS = RS * EY, NP = 2 * R + 1;
    static constexpr int NE = (EX * EY + TILE_T - 1) / TILE_T;  // plane elements per thread
};

// the plane elements a thread moves from global to shared memory: fixed for the whole march
template <typename T, int R>
struct PlaneMap {
    int gofs[T::NE];   // offset inside a (H, W) plane, or -1 outside the volume
    int sofs[T::NE];   // offset inside a shared-memory plane, or -1 for no element
    __device__ __forceinline__ void init(int x0t, int y0t, IrsDims d) {
#pragma unroll
        for (int k = 0; k < T::NE; ++k) {
            const int e = threadIdx.x + k * TILE_T;
            const int ey = e / T::EX, ex = e - ey * T::EX;
            const int gx = x0t - R + ex, gy = y0t - R + ey;
            const bool valid = e < T::EX * T::EY;
            gofs[k] = (valid && gx >= 0 && gx < d.W && gy >= 0 && gy < d.H) ? gy * d.W + gx : -1;
            sofs[k] = valid ? ey * T::RS + ex : -1;
        }
    }
};

template <typename T, int R, int NCH>
__device__ __forceinline__ void plane_fetch(const PlaneMap<T, R>& m, const float* __restrict__ src, long long V, int pz,
                                            IrsDims d, float scale, float (&reg)[NCH][T::NE]) {
    const bool zin = pz >= 0 && pz < d.D;
    const int zofs = pz * d.H * d.W;   // 3 V < 2^31 (IRS_CHECK_DIMS): 32-bit element offsets
    const int Vi = (int)V;
#pragma unroll
    for (int k = 0; k < T::NE; ++k) {
        const bool ok = zin && m.gofs[k] >= 0;
        const int o = zofs + m.gofs[k];
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) reg[ch][k] = ok ? __ldg(src + (ch * Vi + o)) * scale : 0.f;
    }
}

template <typename T, int NCH>
__device__ __forceinline__ bool plane_nonzero(const float (&reg)[NCH][T::NE]) {
    bool nz = false;
#pragma unroll
    for (int k = 0; k < T::NE; ++k)
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) nz = nz || (reg[ch][k] != 0.f);
    return nz;
}

template <typename T, int R, int NCH>
__device__ __forceinline__ void plane_store(const PlaneMap<T, R>& m, float* __restrict__ dst, int ch_stride,
                                            const float (&reg)[NCH][T::NE]) {
#pragma unroll
    for (int k = 0; k < T::NE; ++k) {
        if (m.sofs[k] >= 0) {
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) dst[ch * ch_stride + m.sofs[k]] = reg[ch][k];
        }
    }
}

// trilinear cell in the ring: index of the (x0,y0,z0) corner and the z-corner offset; x/y corner offsets are 1 and EX.
// slot_z = ring slot of plane z (the thread's own plane); the cell's planes lie within z-R .. z+R.
template <typename T, int R>
__device__ __forceinline__ void ring_cell(float px, float py, float pz, int x0t, int y0t, int z, int slot_z, int& i000,
                                          int& sz, float& fx, float& fy, float& fz) {
    const float x0 = floorf(px), y0 = floorf(py), z0 = floorf(pz);
    fx = px - x0; fy = py - y0; fz = pz - z0;
    const int ix = (int)x0, iy = (int)y0, iz = (int)z0;
    int s0 = slot_z + (iz - z);
    s0 += s0 < 0 ? T::NP : 0;
    s0 -= s0 >= T::NP ? T::NP : 0;
    const int s1 = (s0 + 1 == T::NP) ? 0 : s0 + 1;
    i000 = s0 * T::PS + (iy - (y0t - R)) * T::RS + (ix - (x0t - R));
    sz = (s1 - s0) * T::PS;
}

template <int EX>
__device__ __forceinline__ float ring_interp(const float* __restrict__ U, int i, int sz, float fx, float fy, float fz) {
    const float v000 = U[i], v001 = U[i + 1], v010 = U[i + EX], v011 = U[i + EX + 1];
    const float* U1 = U + sz;
    const float v100 = U1[i], v101 = U1[i + 1], v110 = U1[i + EX], v111 = U1[i + EX + 1];
    const float a00 = v000 + fx * (v001 - v000), a01 = v010 + fx * (v011 - v010);
    const float a10 = v100 + fx * (v101 - v100), a11 = v110 + fx * (v111 - v110);
    const float b0 = a00 + fy * (a01 - a00), b1 = a10 + fy * (a11 - a10);
    return b0 + fz * (b1 - b0);
}

template <int EX>
__device__ __forceinline__ void ring_interp_grad(const float* __restrict__ U, int i, int sz, float fx, float fy, float fz,
                                                 float& gx, float& gy, float& gz) {
    const float v000 = U[i], v001 = U[i + 1], v010 = U[i + EX], v011 = U[i + EX + 1];
    const float* U1 = U + sz;
    const float v100 = U1[i], v101 = U1[i + 1], v110 = U1[i + EX], v111 = U1[i + EX + 1];
    const float d00 = v001 - v000, d01 = v011 - v010, d10 = v101 - v100, d11 = v111 - v110;
    const float a00 = v000 + fx * d00, a01 = v010 + fx * d01, a10 = v100 + fx * d10, a11 = v110 + fx * d11;
    const float e0 = a01 - a00, e1 = a11 - a10;
    const float b0 = a00 + fy * e0, b1 = a10 + fy * e1;
    const float dx0 = d00 + fy * (d01 - d00), dx1 = d10 + fy * (d11 - d10);
    gx = dx0 + fz * (dx1 - dx0);
    gy = e0 + fz * (e1 - e0);
    gz = b1 - b0;
}

// packed fp32 pair FMA (Blackwell FFMA2): d = a * b + c on both halves, one issue slot
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}

__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
// scalar x pair (+ pair): ptxas folds the duplicated scalar into the .F32 broadcast operand of FFMA2 / FMUL2
__device__ __forceinline__ float2 ffma2s(float s, float2 b, float2 c) { return ffma2(make_float2(s, s), b, c); }
__device__ __forceinline__ float2 fmul2s(float s, float2 b) { return fmul2(make_float2(s, s), b); }

// position term of the adjoint: sum_c g_c * grad trilinear[u_c](p).  Interpolation is linear in the corner values, so
// the three components are combined at the eight corners first (w = g . u) and ONE gradient is interpolated.
template <int RS>
__device__ __forceinline__ void ring_interp_grad_dot(const float* __restrict__ U, int ch_stride, int i, int sz, float g0,
                                                     float g1, float g2, float fx, float fy, float fz, float& jx,
                                                     float& jy, float& jz) {
    const float* U1 = U + ch_stride;
    const float* U2 = U + 2 * ch_stride;
#define IRS_W(o) (g0 * U[(o)] + g1 * U1[(o)] + g2 * U2[(o)])
    const float v000 = IRS_W(i), v001 = IRS_W(i + 1), v010 = IRS_W(i + RS), v011 = IRS_W(i + RS + 1);
    const float v100 = IRS_W(i + sz), v101 = IRS_W(i + sz + 1), v110 = IRS_W(i + sz + RS), v111 = IRS_W(i + sz + RS + 1);
#undef IRS_W
    const float d00 = v001 - v000, d01 = v011 - v010, d10 = v101 - v100, d11 = v111 - v110;
    const float a00 = v000 + fx * d00, a01 = v010 + fx * d01, a10 = v100 + fx * d10, a11 = v110 + fx * d11;
    const float e0 = a01 - a00, e1 = a11 - a10;
    const float b0 = a00 + fy * e0, b1 = a10 + fy * e1;
    const float dx0 = d00 + fy * (d01 - d00), dx1 = d10 + fy * (d11 - d10);
    jx = dx0 + fz * (dx1 - dx0);
    jy = e0 + fz * (e1 - e0);
    jz = b1 - b0;
}

// ---- forward step -----------------------------------------------------------------------------------------------------
// Threads whose displacement stays inside the ring window (|u| < R) gather from shared memory; the others (large
// deformations) fall back to the global gather, so the kernel is exact for any field.
// block maximum of the per-thread max |u| -> one order-independent atomic per CTA
__device__ __forceinline__ void block_max_to_global(float m, float* __restrict__ maxabs) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float sm[TILE_T / 32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float mm = sm[0];
        for (int w = 1; w < TILE_T / 32; ++w) mm = fmaxf(mm, sm[w]);
        if (mm > 0.f) atomic_max_nonneg(maxabs, mm);
    }
}

template <int R, bool PAD = true>
__device__ __forceinline__ float svf_fwd_tile_body(const float* __restrict__ in, float in_scale, float* __restrict__ out,
                                                   IrsDims d, int x0t, int y0t, int zs, int ze, float* smem) {
    using T = Tile<R, PAD>;
    float* U = smem;  // [3][NP][PS]
    const long long V = d.V();
    const int lx = threadIdx.x % TILE_X, ly = threadIdx.x / TILE_X, x = x0t + lx, y = y0t + ly;
    const bool active = x < d.W && y < d.H;
    const int lc = (ly + R) * T::RS + lx + R;
    const float xmax = (float)(d.W - 1), ymax = (float)(d.H - 1), zmax = (float)(d.D - 1);

    PlaneMap<T, R> map;
    map.init(x0t, y0t, d);
    float reg[3][T::NE];
    for (int pz = zs - R; pz <= zs + R; ++pz) {
        plane_fetch<T, R, 3>(map, in, V, pz, d, in_scale, reg);
        plane_store<T, R, 3>(map, U + (((pz % T::NP) + T::NP) % T::NP) * T::PS, T::NP * T::PS, reg);
    }
    __syncthreads();

    float m = 0.f;
    int slot = zs % T::NP;                       // ring slot of plane z
    int slot_in = (zs + R + 1) % T::NP;          // ring slot the prefetched plane z+R+1 goes to (= slot of plane z-R)
    int gi = (zs * d.H + y) * d.W + x;
    const int HW = d.H * d.W, Vi = (int)V;
    for (int z = zs; z < ze; ++z) {
        plane_fetch<T, R, 3>(map, in, V, z + R + 1, d, in_scale, reg);  // in flight while this plane is processed
        if (active) {
            const float* Uz = U + slot * T::PS + lc;
            const float ux = Uz[0], uy = Uz[T::NP * T::PS], uz = Uz[2 * T::NP * T::PS];
            const float amax = fmaxf(fabsf(ux), fmaxf(fabsf(uy), fabsf(uz)));
            m = fmaxf(m, amax);
            if (amax < (float)R) {
                const float px = irs_clampf((float)x + ux, 0.f, xmax), py = irs_clampf((float)y + uy, 0.f, ymax),
                            pz = irs_clampf((float)z + uz, 0.f, zmax);
                int i000, sz;
                float fx, fy, fz;
                ring_cell<T, R>(px, py, pz, x0t, y0t, z, slot, i000, sz, fx, fy, fz);
                out[gi] = ux + ring_interp<T::RS>(U, i000, sz, fx, fy, fz);
                out[Vi + gi] = uy + ring_interp<T::RS>(U + T::NP * T::PS, i000, sz, fx, fy, fz);
                out[2 * Vi + gi] = uz + ring_interp<T::RS>(U + 2 * T::NP * T::PS, i000, sz, fx, fy, fz);
            } else {
                irs_body_svf_fwd(in, in_scale, out, V, gi, d);
            }
        }
        __syncthreads();  // plane z-R is no longer needed
        plane_store<T, R, 3>(map, U + slot_in * T::PS, T::NP * T::PS, reg);
        __syncthreads();
        slot = slot + 1 == T::NP ? 0 : slot + 1;
        slot_in = slot_in + 1 == T::NP ? 0 : slot_in + 1;
        gi += HW;
    }
    return m;
}

template <int R>
__global__ void __launch_bounds__(TILE_T)
svf_step_fwd_tile_kernel(const float* __restrict__ in_all, float in_scale, float* __restrict__ out_all,
                         float* __restrict__ maxabs, int seg_len, IrsDims d) {
    extern __shared__ __align__(128) float smem[];
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    const long long V = d.V();
    const int tiles_x = (d.W + TILE_X - 1) / TILE_X, tiles_y = (d.H + TILE_Y - 1) / TILE_Y;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int x0t = bx * TILE_X, y0t = by * TILE_Y, zs = bz * seg_len, ze = min(zs + seg_len, d.D);
    const float m = svf_fwd_tile_body<R>(in_all + (size_t)blockIdx.y * 3 * V, in_scale, out_all + (size_t)blockIdx.y * 3 * V,
                                         d, x0t, y0t, zs, ze, smem);
    block_max_to_global(m, maxabs);
}

// ---- adjoint step -------------------------------------------------------------------------------------------------------
// Every source voxel of plane s is visited once per in-plane offset (ox, oy) and deposits into the 2R+1 register
// accumulators of the target planes s-R..s+R: (2R+1)^2 candidates per voxel instead of (2R+1)^3, all from shared memory.
// BORDER = false for tiles whose halo lies strictly inside the volume: positions cannot be clamped there.
template <int R, bool BORDER>
__device__ __forceinline__ void svf_bwd_tile_body(const float* __restrict__ u, float in_scale,
                                                  const float* __restrict__ gp, float* __restrict__ g, float out_scale,
                                                  IrsDims d, int x0t, int y0t, int zs, int ze, float* smem) {
    using T = Tile<R>;
    constexpr int NP = T::NP, PS = T::PS, EX = T::RS;
    float* U = smem;                // [3][NP][PS]  velocity ring, slot = plane mod NP (scaled)
    float* G = smem + 3 * NP * PS;  // [3][PS]      incoming gradient of the current source plane
    // per-row "incoming gradient is non-zero" flags of the current / next source plane: the gradient vanishes outside the
    // (dilated) fixed mask, and a warp (= one row of targets) whose three source rows are all zero skips the transpose
    __shared__ int row_nz[2][T::EY];
    const long long V = d.V();
    const int Vi = (int)V, HW = d.H * d.W;
    const int lx = threadIdx.x % TILE_X, ly = threadIdx.x / TILE_X, x = x0t + lx, y = y0t + ly;
    const bool active = x < d.W && y < d.H;
    const int lc = (ly + R) * EX + lx + R;
    const float xf = (float)x, yf = (float)y;
    const float xmax = (float)(d.W - 1), ymax = (float)(d.H - 1), zmax = (float)(d.D - 1);

    PlaneMap<T, R> map;
    map.init(x0t, y0t, d);
    float ru[3][T::NE], rg[3][T::NE];
    const int s_first = zs - R, s_last = ze - 1 + R;
    for (int pz = s_first - R; pz <= s_first + R; ++pz) {
        plane_fetch<T, R, 3>(map, u, V, pz, d, in_scale, ru);
        plane_store<T, R, 3>(map, U + (((pz % NP) + NP) % NP) * PS, NP * PS, ru);
    }
    auto flag_rows = [&](int buf) {
#pragma unroll
        for (int k = 0; k < T::NE; ++k) {
            if (map.sofs[k] >= 0 && (rg[0][k] != 0.f || rg[1][k] != 0.f || rg[2][k] != 0.f)) row_nz[buf][map.sofs[k] / T::RS] = 1;
        }
    };
    if (threadIdx.x < 2 * T::EY) row_nz[threadIdx.x / T::EY][threadIdx.x % T::EY] = 0;
    __syncthreads();
    plane_fetch<T, R, 3>(map, gp, V, s_first, d, 1.f, rg);
    plane_store<T, R, 3>(map, G, PS, rg);
    int cur = 0;
    flag_rows(cur);
    // planes of a tile whose incoming gradient is entirely zero are skipped altogether
    bool g_nonzero = __syncthreads_or(plane_nonzero<T, 3>(rg));

    float2 acc01[NP];   // components x, y of the 2R+1 target planes (packed: updated with FFMA2)
    float acc2[NP];     // component z
#pragma unroll
    for (int i = 0; i < NP; ++i) { acc01[i] = make_float2(0.f, 0.f); acc2[i] = 0.f; }

    int slot = ((s_first % NP) + NP) % NP;             // ring slot of source plane s
    int slot_in = (((s_first + R + 1) % NP) + NP) % NP;  // where the prefetched plane s+R+1 goes (= slot of plane s-R)
    int gi = ((s_first - R) * d.H + y) * d.W + x;       // index of target (x, y, s-R)
    for (int s = s_first; s <= s_last; ++s) {
        plane_fetch<T, R, 3>(map, u, V, s + R + 1, d, in_scale, ru);   // in flight while plane s is processed
        plane_fetch<T, R, 3>(map, gp, V, s + 1, d, 1.f, rg);
        if (threadIdx.x < T::EY) row_nz[cur ^ 1][threadIdx.x] = 0;   // last read before the previous barrier pair
        bool rows_nz = false;
#pragma unroll
        for (int oy = -R; oy <= R; ++oy) rows_nz = rows_nz || (row_nz[cur][ly + R + oy] != 0);
        if (g_nonzero && active && s >= 0 && s < d.D) {
            const float* Us = U + slot * PS;
            const float sf = (float)s;
            // ---- interpolation transpose ----
            if (rows_nz) {
#pragma unroll
            for (int oy = -R; oy <= R; ++oy) {
                if (BORDER && (y + oy < 0 || y + oy >= d.H)) continue;
#pragma unroll
                for (int ox = -R; ox <= R; ++ox) {
                    if (BORDER && (x + ox < 0 || x + ox >= d.W)) continue;
                    const int li = lc + oy * EX + ox;
                    float cx = Us[li], cy = Us[NP * PS + li];
                    if (BORDER) {  // clamp(s + u) - s
                        cx = irs_clampf(cx, -(xf + (float)ox), xmax - (xf + (float)ox));
                        cy = irs_clampf(cy, -(yf + (float)oy), ymax - (yf + (float)oy));
                    }
                    float wx, wy;
                    if (R == 1) {  // |c| < 1: the hat function reduces to one max / one subtraction
                        wx = ox < 0 ? fmaxf(cx, 0.f) : (ox > 0 ? fmaxf(-cx, 0.f) : 1.f - fabsf(cx));
                        wy = oy < 0 ? fmaxf(cy, 0.f) : (oy > 0 ? fmaxf(-cy, 0.f) : 1.f - fabsf(cy));
                    } else {
                        wx = fmaxf(0.f, 1.f - fabsf(cx + (float)ox));
                        wy = fmaxf(0.f, 1.f - fabsf(cy + (float)oy));
                    }
                    const float wxy = wx * wy;
                    float cz = Us[2 * NP * PS + li];
                    if (BORDER) cz = irs_clampf(cz, -sf, zmax - sf);
                    const float2 g01 = make_float2(G[li], G[PS + li]);
                    const float g2 = G[2 * PS + li];
                    if (R == 1) {
                        const float wm = wxy * fmaxf(-cz, 0.f), w0 = wxy * (1.f - fabsf(cz)), wp = wxy * fmaxf(cz, 0.f);
                        acc01[0] = ffma2(make_float2(wm, wm), g01, acc01[0]); acc2[0] += wm * g2;
                        acc01[1] = ffma2(make_float2(w0, w0), g01, acc01[1]); acc2[1] += w0 * g2;
                        acc01[2] = ffma2(make_float2(wp, wp), g01, acc01[2]); acc2[2] += wp * g2;
                    } else {
                        if (wxy == 0.f) continue;
#pragma unroll
                        for (int dz = -R; dz <= R; ++dz) {
                            const float w = wxy * fmaxf(0.f, 1.f - fabsf(cz - (float)dz));
                            acc01[dz + R] = ffma2(make_float2(w, w), g01, acc01[dz + R]); acc2[dz + R] += w * g2;
                        }
                    }
                }
            }
            }
            // ---- direct + position term of target (x, y, s) ----
            if (s >= zs && s < ze && row_nz[cur][ly + R] != 0) {
                const float g0 = G[lc], g1 = G[PS + lc], g2 = G[2 * PS + lc];
                float px = xf + Us[lc], py = yf + Us[NP * PS + lc], pz = sf + Us[2 * NP * PS + lc];
                float mx = 1.f, my = 1.f, mz = 1.f;
                if (BORDER) {
                    mx = irs_inside(px, d.W); my = irs_inside(py, d.H); mz = irs_inside(pz, d.D);
                    px = irs_clampf(px, 0.f, xmax); py = irs_clampf(py, 0.f, ymax); pz = irs_clampf(pz, 0.f, zmax);
                }
                int i000, sz;
                float fx, fy, fz, jx, jy, jz;
                ring_cell<T, R>(px, py, pz, x0t, y0t, s, slot, i000, sz, fx, fy, fz);
                ring_interp_grad_dot<T::RS>(U, NP * PS, i000, sz, g0, g1, g2, fx, fy, fz, jx, jy, jz);
                acc01[R].x += g0 + mx * jx; acc01[R].y += g1 + my * jy; acc2[R] += g2 + mz * jz;
            }
        }
        // ---- target plane s-R is complete ----
        if (active && s - R >= zs && s - R < ze) {
            g[gi] = acc01[0].x * out_scale; g[Vi + gi] = acc01[0].y * out_scale; g[2 * Vi + gi] = acc2[0] * out_scale;
        }
#pragma unroll
        for (int i = 0; i < NP - 1; ++i) { acc01[i] = acc01[i + 1]; acc2[i] = acc2[i + 1]; }
        acc01[NP - 1] = make_float2(0.f, 0.f); acc2[NP - 1] = 0.f;
        __syncthreads();                 // everyone is done with ring plane s-R and with G
        plane_store<T, R, 3>(map, U + slot_in * PS, NP * PS, ru);
        plane_store<T, R, 3>(map, G, PS, rg);
        cur ^= 1;
        flag_rows(cur);
        g_nonzero = __syncthreads_or(plane_nonzero<T, 3>(rg));
        slot = slot + 1 == NP ? 0 : slot + 1;
        slot_in = slot_in + 1 == NP ? 0 : slot_in + 1;
        gi += HW;
    }
}

// tile path of one adjoint step for gather radius R (from the step's max |u|): R = 1 / 2 from shared-memory rings, wider
// windows straight from global memory; beyond radius_max only the direct + position terms (the scatter kernel that
// follows adds the interpolation transpose with atomics)
__device__ __forceinline__ void svf_bwd_tile_dispatch(int R, const float* __restrict__ in, float in_scale,
                                                      const float* __restrict__ gp, float* __restrict__ g, int radius_max,
                                                      float out_scale, IrsDims d, int x0t, int y0t, int zs, int ze,
                                                      float* smem) {
    // the tile, its halo and every clamped position stay strictly inside the volume?
    auto interior = [&](int Rr) {
        return x0t - 2 * Rr >= 0 && x0t + TILE_X - 1 + 2 * Rr <= d.W - 1 && y0t - 2 * Rr >= 0 &&
               y0t + TILE_Y - 1 + 2 * Rr <= d.H - 1 && zs - 2 * Rr >= 0 && ze - 1 + 2 * Rr <= d.D - 1;
    };
    if (R <= radius_max && R == 1) {
        if (interior(1)) svf_bwd_tile_body<1, false>(in, in_scale, gp, g, out_scale, d, x0t, y0t, zs, ze, smem);
        else svf_bwd_tile_body<1, true>(in, in_scale, gp, g, out_scale, d, x0t, y0t, zs, ze, smem);
    } else if (R <= radius_max && R == 2) {
        svf_bwd_tile_body<2, true>(in, in_scale, gp, g, out_scale, d, x0t, y0t, zs, ze, smem);
    } else {
        const int x = x0t + (threadIdx.x % TILE_X), y = y0t + (threadIdx.x / TILE_X);
        if (x >= d.W || y >= d.H) return;
        const long long V = d.V();
        for (int z = zs; z < ze; ++z)
            irs_body_svf_bwd(in, in_scale, gp, g, R <= radius_max ? R : -1, out_scale, V,
                             ((long long)z * d.H + y) * d.W + x, d);
    }
}

// out-of-line copy for kernels whose main path is another one: keeps the fallback's register pressure out of it
__device__ __noinline__ void svf_bwd_tile_dispatch_cold(int R, const float* __restrict__ in, float in_scale,
                                                        const float* __restrict__ gp, float* __restrict__ g, int radius_max,
                                                        float out_scale, IrsDims d, int x0t, int y0t, int zs, int ze,
                                                        float* smem) {
    svf_bwd_tile_dispatch(R, in, in_scale, gp, g, radius_max, out_scale, d, x0t, y0t, zs, ze, smem);
}

// Radius a tile may use: the step's global radius R, or 1 when every source within R voxels of the tile's targets moves by
// less than one voxel (sources farther away cannot reach it: they move by less than R).  Only in the gather regime
// (2 <= R <= radius_max): beyond it the scatter companion adds the whole transpose and tiles must not do their own.
__device__ __forceinline__ int svf_local_radius(int R, int radius_max, const IrsCells& cm, int chain, int x0t, int y0t, int ty,
                                                int zs, int ze) {
    if (R < 2 || R > radius_max || cm.p == nullptr) return R;
    const float m = cells_region_max(cm, chain, x0t - R, x0t + TILE_X - 1 + R, y0t - R, y0t + ty - 1 + R, zs - R, ze - 1 + R);
    return m < 0.999f ? 1 : R;
}

// gather radius of a step from its max |u|.  The R = 1 kernels assume that x + u never ROUNDS to x +- 1 in fp32, hence the
// margin (ulp(x) / 2 < 1e-3 for every supported volume size).
__device__ __forceinline__ int svf_gather_radius(float maxabs) { return (int)floorf(maxabs + 1e-3f) + 1; }

__global__ void __launch_bounds__(TILE_T, 4)
svf_step_bwd_tile_kernel(const float* __restrict__ in, float in_scale, const float* __restrict__ gp_all,
                         float* __restrict__ g_all, const float* __restrict__ maxabs, int radius_max, float out_scale,
                         int seg_len, IrsDims d, IrsCells cm) {
    extern __shared__ __align__(128) float smem[];
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    int R = svf_gather_radius(__ldg(maxabs));
    const long long V = d.V();
    const size_t off = (size_t)blockIdx.y * 3 * V;
    const int tiles_x = (d.W + TILE_X - 1) / TILE_X, tiles_y = (d.H + TILE_Y - 1) / TILE_Y;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int x0t = bx * TILE_X, y0t = by * TILE_Y, zs = bz * seg_len, ze = min(zs + seg_len, d.D);
    R = svf_local_radius(R, radius_max, cm, blockIdx.y, x0t, y0t, TILE_Y, zs, ze);
    svf_bwd_tile_dispatch(R, in + off, in_scale, gp_all + off, g_all + off, radius_max, out_scale, d, x0t, y0t, zs, ze, smem);
}

// ---------------------------------------------------------------------------------------------------------------------
// TMA-fed kernels for steps with max |u| < 1 (every step of a typical registration; the rings above remain the path for
// larger displacements and for row pitches the TMA unit cannot address).  One thread issues ONE cp.async.bulk.tensor per
// z-plane (tile + halo 1, three components, zeros outside the volume) into a 4-slot shared-memory ring guarded by
// mbarriers; nobody spends issue slots on global loads, address arithmetic or bounds predicates.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TMA_EX = TILE_X + 2, TMA_EY = TILE_Y + 2;   // valid tile + halo 1
constexpr int TMA_NS = 4;                                  // ring slots: planes z-1, z, z+1 and one in flight
constexpr int TMA_XO = 4;   // the TMA unit wants a 16-byte aligned innermost coordinate: boxes start at x0t - 4 (measured:
                            // an unaligned start raises "illegal instruction"); column TMA_XO of a box is the tile's x0t

template <int BW>   // box width = shared-memory row stride (floats); BW * 4 bytes must be a multiple of 16
struct TmaRing {
    static_assert(BW >= TMA_XO + TILE_X + 2 && (BW * 4) % 16 == 0, "box width");
    static constexpr int CS = TMA_EY * BW;                              // component stride
    static constexpr uint32_t BYTES = 3u * CS * 4u;                     // one plane box
    static constexpr int SS = (int)((BYTES + 127u) / 128u * 128u / 4u); // slot stride (floats), 128-byte aligned
};

// trilinear cell in a TMA ring: q0 = ring sequence number of plane floor(pz) (slot = q & 3)
template <int BW>
__device__ __forceinline__ void tma_ring_cell(float px, float py, float pz, int x0t, int y0t, int z, int q_z, int& i000,
                                              int& sz, float& fx, float& fy, float& fz) {
    using RG = TmaRing<BW>;
    const float x0 = floorf(px), y0 = floorf(py), z0 = floorf(pz);
    fx = px - x0; fy = py - y0; fz = pz - z0;
    const int ix = (int)x0, iy = (int)y0, iz = (int)z0;
    const int s0 = (q_z + (iz - z)) & (TMA_NS - 1), s1 = (s0 + 1) & (TMA_NS - 1);
    i000 = s0 * RG::SS + (iy - (y0t - 1)) * BW + (ix - (x0t - TMA_XO));
    sz = (s1 - s0) * RG::SS;
}

// exact global gather for one voxel, out of line: its register pressure stays out of the TMA kernels' main path
__device__ __noinline__ void svf_fwd_voxel_cold(const float* __restrict__ in, float in_scale, float* __restrict__ out,
                                                long long V, long long i, IrsDims d) {
    irs_body_svf_fwd(in, in_scale, out, V, i, d);
}

// ---- forward step ------------------------------------------------------------------------------------------------------
// voxels with |u| >= 0.999 (rare; only the last steps of a large deformation) take the exact global gather
// ENERGY: the regulariser energy of the (unscaled) input field -- sum over components and axes of squared forward
// differences, last difference counted twice (reference model/loss.py:152-161, utils/diff_op.py:83-96) -- accumulated
// from the ring into `energy_acc`: every neighbour it needs is already in shared memory.
template <int BW, bool ENERGY>
__device__ __forceinline__ float svf_fwd_tma_body(const CUtensorMap* tmap, const float* __restrict__ in, float in_scale,
                                                  float* __restrict__ out, IrsDims d, int chain, int x0t, int y0t, int zs,
                                                  int ze, float* smem, float& energy_acc) {
    using RG = TmaRing<BW>;
    float* U = smem;                                                           // [4 slots][3][EY][BW]
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + TMA_NS * RG::SS);      // one mbarrier per slot
    const int tid = threadIdx.x;
    const int lx = tid % TILE_X, ly = tid / TILE_X, x = x0t + lx, y = y0t + ly;
    const bool active = x < d.W && y < d.H;
    const int lc = (ly + 1) * BW + lx + TMA_XO;
    const float xmax = (float)(d.W - 1), ymax = (float)(d.H - 1), zmax = (float)(d.D - 1);
    const long long V = d.V();
    const int Vi = (int)V, HW = d.H * d.W;
    const int n_planes = (ze - zs) + 2;   // planes zs-1 .. ze, ring sequence number q = plane - (zs - 1)

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < TMA_NS; ++i) irs_mbar_init(&bar[i], 1);
        irs_mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0) {
        for (int q = 0; q < TMA_NS && q < n_planes; ++q) {
            irs_mbar_expect_tx(&bar[q], RG::BYTES);
            irs_tma_load_plane(U + q * RG::SS, tmap, &bar[q], x0t - TMA_XO, y0t - 1, zs - 1 + q, 3 * chain);
        }
    }
    float m = 0.f;
    int gi = (zs * d.H + y) * d.W + x;
    irs_mbar_wait(&bar[0], 0);
    irs_mbar_wait(&bar[1], 0);
    for (int z = zs, it = 0; z < ze; ++z, ++it) {
        irs_mbar_wait(&bar[(it + 2) & 3], ((it + 2) >> 2) & 1);   // plane z+1 has landed
        if (active) {
            const float* Uz = U + ((it + 1) & 3) * RG::SS + lc;
            if (ENERGY) {
                const float* Un = U + ((it + 2) & 3) * RG::SS + lc;   // plane z+1
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) {
                    const float c0 = Uz[ch * RG::CS];
                    energy_acc += irs_diff_energy(c0, Uz[ch * RG::CS + 1], x, d.W) + irs_diff_energy(c0, Uz[ch * RG::CS + BW], y, d.H) +
                                  irs_diff_energy(c0, Un[ch * RG::CS], z, d.D);
                }
            }
            const float ux = Uz[0] * in_scale, uy = Uz[RG::CS] * in_scale, uz = Uz[2 * RG::CS] * in_scale;
            const float amax = fmaxf(fabsf(ux), fmaxf(fabsf(uy), fabsf(uz)));
            m = fmaxf(m, amax);
            if (amax < 0.999f) {
                const float px = irs_clampf((float)x + ux, 0.f, xmax), py = irs_clampf((float)y + uy, 0.f, ymax),
                            pz = irs_clampf((float)z + uz, 0.f, zmax);
                int i000, sz;
                float fx, fy, fz;
                tma_ring_cell<BW>(px, py, pz, x0t, y0t, z, it + 1, i000, sz, fx, fy, fz);
                // interpolation is linear in the samples and in_scale is a power of two: scaling after is bit-identical
                out[gi] = ux + in_scale * ring_interp<BW>(U, i000, sz, fx, fy, fz);
                out[Vi + gi] = uy + in_scale * ring_interp<BW>(U + RG::CS, i000, sz, fx, fy, fz);
                out[2 * Vi + gi] = uz + in_scale * ring_interp<BW>(U + 2 * RG::CS, i000, sz, fx, fy, fz);
            } else {
                svf_fwd_voxel_cold(in, in_scale, out, V, gi, d);
            }
        }
        __syncthreads();   // everyone is done with plane z-1: its slot takes plane z+3
        if (tid == 0 && it + 4 < n_planes) {
            irs_mbar_expect_tx(&bar[it & 3], RG::BYTES);
            irs_tma_load_plane(U + (it & 3) * RG::SS, tmap, &bar[it & 3], x0t - TMA_XO, y0t - 1, zs + 3 + it, 3 * chain);
        }
        gi += HW;
    }
    return m;
}

// Row pitch of the forward step's plane boxes.  64 floats (a multiple of the 32 banks): all rows alias the same banks, so lanes whose
// cells lie in different rows do not collide as long as neighbouring lanes pick the same column offset -- measured 0.2146 -> 0.2112 ms
// for the 12 steps on the benchmark's rank-0 draw and 0.2498 -> 0.2357 ms on a typical draw, although the unit moves 60 % more bytes
// per plane than with the tight pitch of 40.  The adjoint keeps 40: at 64 its two rings no longer fit twice per SM.
constexpr int FWD_BW = 64;
constexpr size_t svf_fwd_tma_smem() { return sizeof(float) * TMA_NS * TmaRing<FWD_BW>::SS + 8 * TMA_NS; }

// out-of-line fallbacks of the TMA forward kernel: their register pressure stays out of the main path
__device__ __noinline__ float svf_fwd_tile_body_cold(const float* __restrict__ in, float in_scale, float* __restrict__ out,
                                                     IrsDims d, int x0t, int y0t, int zs, int ze, float* smem) {
    return svf_fwd_tile_body<2, false>(in, in_scale, out, d, x0t, y0t, zs, ze, smem);   // compact ring (no row padding)
}

constexpr size_t svf_fwd_tile_smem_compact(int R) {
    return sizeof(float) * (size_t)(3 * (2 * R + 1)) * (TILE_X + 2 * R) * (TILE_Y + 2 * R);
}

// maxabs_prev = max |u_{k-1}| of the previous step (nullptr for the first): |u_k| <= 2 max |u_{k-1}|, so the TMA ring is
// taken when that bound is below three voxels (see `small` below), the wider non-TMA ring otherwise
// Compiled for 5 resident CTAs per SM (register cap 65536 / 256 / 5): measured at 128^3, 4 -> 0.212 ms, 5 -> 0.200 ms,
// 6 -> 0.208 ms for the 12 forward steps.  ENERGY (first step only):
// also reduces the regulariser energy of the input field per chain -- block sums in double, partials[blockIdx.x], the
// last block of the chain adds them in block order (deterministic) -> energy[chain * energy_stride].
struct IrsEnergyOut {
    double* energy;          // nullptr: the caller computes the energy itself
    long long energy_stride;
    double* partials;        // gridDim.x doubles per chain
    unsigned int* counters;  // one per chain, zero on entry, reset on exit
};

template <bool ENERGY>
__global__ void __launch_bounds__(TILE_T, 5)
svf_step_fwd_tma_kernel(const __grid_constant__ CUtensorMap tmap, const float* __restrict__ in_all, float in_scale,
                        float* __restrict__ out_all, const float* __restrict__ maxabs_prev, float* __restrict__ maxabs,
                        int seg_len, IrsDims d, IrsEnergyOut eo) {
    extern __shared__ __align__(128) float smem[];
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    const long long V = d.V();
    const int tiles_x = (d.W + TILE_X - 1) / TILE_X, tiles_y = (d.H + TILE_Y - 1) / TILE_Y;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int x0t = bx * TILE_X, y0t = by * TILE_Y, zs = bz * seg_len, ze = min(zs + seg_len, d.D);
    const float* in = in_all + (size_t)blockIdx.y * 3 * V;
    float* out = out_all + (size_t)blockIdx.y * 3 * V;
    // The TMA body is exact for any field: a voxel whose |u| reaches one voxel takes the global gather on its own.  It is the
    // faster choice as long as such voxels are a minority (they are spatially coherent, so whole warps go one way or the other):
    // measured, a step whose bound 2 max|u_{k-1}| just exceeds one voxel cost 3x in the wide-ring kernel although only a few
    // voxels were affected (16 % of the whole forward pass on a 128^3 chain).  Only when the bound says that displacements of
    // several voxels are common does the wide ring (R = 2, then global gathers) take the whole step.
    const bool small = maxabs_prev == nullptr || 2.f * __ldg(maxabs_prev) < 3.0f;   // always true for the first step
    float m, e_acc = 0.f;
    if (small) m = svf_fwd_tma_body<FWD_BW, ENERGY>(&tmap, in, in_scale, out, d, blockIdx.y, x0t, y0t, zs, ze, smem, e_acc);
    else m = svf_fwd_tile_body_cold(in, in_scale, out, d, x0t, y0t, zs, ze, smem);
    block_max_to_global(m, maxabs);
    if (ENERGY) {
        __shared__ double sh[32];
        __shared__ double total[1];
        double blk[1];
        __syncthreads();
        irs_block_sum<1>(&e_acc, blk, sh);
        if (irs_grid_sum<1>(blk, eo.partials + (size_t)blockIdx.y * gridDim.x, eo.counters + blockIdx.y, total)) {
            if (threadIdx.x == 0) eo.energy[(size_t)blockIdx.y * eo.energy_stride] = total[0];
        }
    }
}

// ---- adjoint step ------------------------------------------------------------------------------------------------------
// Per source plane s the CTA first turns every source voxel of the tile + halo into a RECORD
//     { cx, cy, g0, g1 } { g2, wz_0, wz_1, wz_2 }                 two 128-bit shared-memory words (in two arrays)
// where (cx, cy, cz) = clamp(s + u(s)) - s is the source's sub-voxel offset, g = dL/du_{k+1}(s), and wz_0..2 are its hat
// weights onto the target planes s-1, s and s+1.  A target then needs, per in-plane neighbour, two LDS.128, two weight ops
// and the products with the record -- the z weights and the border clamps are paid once per source instead of nine times.
// (A 12-float record holding the nine products wz_b * g_c saves four instructions per neighbour but costs a third
// LDS.128: measured shared-memory bound, 61 % of the LSU data pipe vs 50 % issue.)
// The tile is 32 x 16: thread (lx, ly) owns the targets in rows 2 ly and 2 ly + 1, whose neighbourhoods share two of their
// three source rows -- against one target per thread, 12 record loads for two targets instead of 18, half the barriers and
// TMA issues per voxel, a smaller halo share (34 x 18 records for 512 targets).  128 registers, 2 CTAs per SM.
constexpr int REC_F = 8;    // floats per record
constexpr int BWD_NG = 3;   // ring slots of the incoming gradient: plane s and two in flight (slot = plane mod 3, static)
constexpr int BWD_BW = 40;  // row pitch of the plane boxes (why not 64: see FWD_BW)
constexpr int B2_TY = 16, B2_EY = B2_TY + 2, B2_NR = TMA_EX * B2_EY;                  // 612 records per plane
constexpr int B2_CS = B2_EY * BWD_BW;                                               // component stride of a plane box
constexpr uint32_t B2_BYTES = 3u * B2_CS * 4u;
constexpr int B2_SS = (int)((B2_BYTES + 127u) / 128u * 128u / 4u);                  // slot stride (floats)
constexpr size_t svf_bwd_tma2_smem() {
    return sizeof(float) * ((TMA_NS + BWD_NG) * B2_SS + 2 * B2_NR * REC_F) + 8 * (TMA_NS + BWD_NG) + 4 * 3 * B2_EY + 8;
}

struct BwdTmaCtx {
    const CUtensorMap *tmap_u, *tmap_g;
    float *U, *G, *REC;
    int* row_nz;          // [3][B2_EY]: "this source row has a non-zero gradient", per plane modulo 3
    uint64_t *bar_u, *bar_g;
    float in_scale, out_scale;
    IrsDims d;
    int x0t, y0t, zs, ze, chain;
    float* g;
};

// |c| < 1: hat weight of a source at in-plane offset o (-1, 0, 1; constant-folded) onto the target column
__device__ __forceinline__ float hat_small_rt(float c, int o) {
    return o < 0 ? fmaxf(c, 0.f) : (o > 0 ? fmaxf(-c, 0.f) : 1.f - fabsf(c));
}

__device__ __forceinline__ void svf_bwd_tma2_body(const BwdTmaCtx& c) {
    constexpr int BW = BWD_BW, CS = B2_CS, SS = B2_SS, NRP = (B2_NR + TILE_T - 1) / TILE_T;   // 3 records per thread
    const int tid = threadIdx.x;
    const IrsDims d = c.d;
    const int lx = tid % TILE_X, ly = tid / TILE_X, x = c.x0t + lx;
    const int ty0 = 2 * ly;                                   // tile row of target 0 (target 1 = ty0 + 1)
    const int y0 = c.y0t + ty0;
    const bool act[2] = {x < d.W && y0 < d.H, x < d.W && y0 + 1 < d.H};
    const int lc0 = (ty0 + 1) * BW + lx + TMA_XO;             // target 0 inside a plane box (target 1: + BW)
    const int lr0 = (ty0 + 1) * TMA_EX + lx + 1;              // target 0's record (target 1: + TMA_EX)
    const float xf = (float)x;
    const float xmax = (float)(d.W - 1), ymax = (float)(d.H - 1), zmax = (float)(d.D - 1);
    const int Vi = (int)d.V(), HW = d.H * d.W;
    const int zs = c.zs, ze = c.ze;
    const int s_first = zs - 1, n_it = (ze - zs) + 2;
    const int n_u = n_it + 2, n_g = n_it;

    int rec_e[NRP], rec_po[NRP], rec_row[NRP];
    float rec_lox[NRP], rec_loy[NRP];
#pragma unroll
    for (int k = 0; k < NRP; ++k) {
        const int e = tid + k * TILE_T;
        const int ey = e / TMA_EX, ex = e - ey * TMA_EX;
        rec_e[k] = e < B2_NR ? e : -1;
        rec_po[k] = ey * BW + ex + (TMA_XO - 1);
        rec_row[k] = ey;
        rec_lox[k] = -(float)(c.x0t - 1 + ex);
        rec_loy[k] = -(float)(c.y0t - 1 + ey);
    }

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < TMA_NS; ++i) irs_mbar_init(&c.bar_u[i], 1);
#pragma unroll
        for (int i = 0; i < BWD_NG; ++i) irs_mbar_init(&c.bar_g[i], 1);
        irs_mbar_fence_init();
    }
    if (tid < 3 * B2_EY) c.row_nz[tid] = 0;
    __syncthreads();
    if (tid == 0) {
        for (int q = 0; q < TMA_NS && q < n_u; ++q) {
            irs_mbar_expect_tx(&c.bar_u[q], B2_BYTES);
            irs_tma_load_plane(c.U + q * SS, c.tmap_u, &c.bar_u[q], c.x0t - TMA_XO, c.y0t - 1, zs - 2 + q, 3 * c.chain);
        }
        for (int q = 0; q < BWD_NG && q < n_g; ++q) {
            irs_mbar_expect_tx(&c.bar_g[q], B2_BYTES);
            irs_tma_load_plane(c.G + q * SS, c.tmap_g, &c.bar_g[q], c.x0t - TMA_XO, c.y0t - 1, zs - 1 + q, 3 * c.chain);
        }
    }

    // Bank order of a record's z weights is fixed: {target plane s-1, s, s+1}; the accumulators rotate by register moves
    // once per plane (12 moves) instead of unrolling the plane loop by three -- a third of the code, fewer instruction
    // cache misses (measured 94 % hit rate / 0.31 stall cycles per issue with the unrolled body).
    auto produce = [&](int itp) {
        const int MP = itp % 3;   // ring slot of the gradient plane and of the row flags
        const int s = s_first + itp;
        if (s < 0 || s >= d.D) return;
        const float* Us = c.U + ((itp + 1) & 3) * SS;
        const float* Gs = c.G + MP * SS;
        float4* rec = reinterpret_cast<float4*>(c.REC) + (itp & 1) * (2 * B2_NR);
        const float sf = (float)s;
#pragma unroll
        for (int k = 0; k < NRP; ++k) {
            if (rec_e[k] < 0) continue;
            const int po = rec_po[k];
            const float g0 = Gs[po], g1 = Gs[CS + po], g2 = Gs[2 * CS + po];
            const float cx = irs_clampf(Us[po] * c.in_scale, rec_lox[k], xmax + rec_lox[k]);
            const float cy = irs_clampf(Us[CS + po] * c.in_scale, rec_loy[k], ymax + rec_loy[k]);
            const float cz = irs_clampf(Us[2 * CS + po] * c.in_scale, -sf, zmax - sf);
            const float wm = fmaxf(-cz, 0.f), w0 = 1.f - fabsf(cz), wp = fmaxf(cz, 0.f);
            float4* r = rec + rec_e[k];
            r[0] = make_float4(cx, cy, g0, g1);
            r[B2_NR] = make_float4(g2, wm, w0, wp);
            if (((__float_as_uint(g0) | __float_as_uint(g1) | __float_as_uint(g2)) << 1) != 0u)   // any non-zero (+-0 are zero)
                c.row_nz[MP * B2_EY + rec_row[k]] = 1;
        }
    };

    // Accumulators: XY[j][b] = components (x, y) of target j in bank b; ZZ[b] = component z of targets (0, 1) in bank b.
    // A record of the two source rows that both targets see costs 3 FMUL2 + 9 FFMA2 for its 18 products (the z components of
    // the two targets share one packed FMA); bank 0 = target plane s-1, 1 = s, 2 = s+1, rotated by register moves per plane.
    float2 XY[2][3], ZZ[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) { XY[0][b] = XY[1][b] = ZZ[b] = make_float2(0.f, 0.f); }
    int gi = ((s_first - 1) * d.H + y0) * d.W + x;   // index of target 0 in plane s-1 (target 1: + W)
    irs_mbar_wait(&c.bar_u[0], 0);
    irs_mbar_wait(&c.bar_u[1], 0);
    irs_mbar_wait(&c.bar_g[0], 0);
    produce(0);
    __syncthreads();
    if (tid == 0 && BWD_NG < n_g) {
        irs_mbar_expect_tx(&c.bar_g[0], B2_BYTES);
        irs_tma_load_plane(c.G, c.tmap_g, &c.bar_g[0], c.x0t - TMA_XO, c.y0t - 1, zs - 1 + BWD_NG, 3 * c.chain);
    }

    for (int it = 0; it < n_it; ++it) {
        const int M = it % 3, BP = (it + 1) % 3, BMf = (it + 2) % 3;   // ring slots (gradient planes, row flags)
        const int s = s_first + it;
        irs_mbar_wait(&c.bar_u[(it + 2) & 3], ((it + 2) >> 2) & 1);
        if (tid < B2_EY) c.row_nz[BMf * B2_EY + tid] = 0;
        if (it + 1 < n_it) {
            irs_mbar_wait(&c.bar_g[BP], ((it + 1) / 3) & 1);
            produce(it + 1);
        }
        const float* Us = c.U + ((it + 1) & 3) * SS;
        const float4* rec = reinterpret_cast<const float4*>(c.REC) + (it & 1) * (2 * B2_NR);
        if ((act[0] || act[1]) && s >= 0 && s < d.D) {
            const int* nz = c.row_nz + M * B2_EY + ty0;   // flags of record rows ty0 .. ty0 + 3
            const int nz1 = nz[1], nz2 = nz[2];
            float gown[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
            // A row without gradient adds exact zeros, so the four rows run as ONE straight-line block whenever any of them
            // carries gradient (warp-uniform): the scheduler can overlap the record loads of a row with the previous row's FMAs.
            if ((nz[0] | nz1 | nz2 | nz[3]) != 0) {
#pragma unroll
                for (int ox = -1; ox <= 1; ++ox) {   // row 0: target 0 only (oy = -1); row 3: target 1 only (oy = +1)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float4* r = rec + (lr0 + (e == 0 ? -1 : 2) * TMA_EX + ox);
                        const float4 r0 = r[0], r1 = r[B2_NR];
                        const float w = hat_small_rt(r0.x, ox) * hat_small_rt(r0.y, e == 0 ? -1 : 1);
                        const float2 g01 = make_float2(r0.z, r0.w);
                        const float w0 = w * r1.y, w1 = w * r1.z, w2 = w * r1.w;
                        XY[e][0] = ffma2s(w0, g01, XY[e][0]);
                        XY[e][1] = ffma2s(w1, g01, XY[e][1]);
                        XY[e][2] = ffma2s(w2, g01, XY[e][2]);
                        if (e == 0) { ZZ[0].x = fmaf(w0, r1.x, ZZ[0].x); ZZ[1].x = fmaf(w1, r1.x, ZZ[1].x); ZZ[2].x = fmaf(w2, r1.x, ZZ[2].x); }
                        else        { ZZ[0].y = fmaf(w0, r1.x, ZZ[0].y); ZZ[1].y = fmaf(w1, r1.x, ZZ[1].y); ZZ[2].y = fmaf(w2, r1.x, ZZ[2].y); }
                    }
                }
#pragma unroll
                for (int rr = 1; rr <= 2; ++rr) {    // rows seen by both targets: oy = rr - 1 (target 0), rr - 2 (target 1)
#pragma unroll
                    for (int ox = -1; ox <= 1; ++ox) {
                        const float4* r = rec + (lr0 + (rr - 1) * TMA_EX + ox);
                        const float4 r0 = r[0], r1 = r[B2_NR];
                        const float wx = hat_small_rt(r0.x, ox);
                        const float2 W = fmul2s(wx, make_float2(hat_small_rt(r0.y, rr - 1), hat_small_rt(r0.y, rr - 2)));
                        const float2 g01 = make_float2(r0.z, r0.w);
                        const float2 W0 = fmul2s(r1.y, W), W1 = fmul2s(r1.z, W), W2 = fmul2s(r1.w, W);
                        XY[0][0] = ffma2s(W0.x, g01, XY[0][0]); XY[1][0] = ffma2s(W0.y, g01, XY[1][0]); ZZ[0] = ffma2s(r1.x, W0, ZZ[0]);
                        XY[0][1] = ffma2s(W1.x, g01, XY[0][1]); XY[1][1] = ffma2s(W1.y, g01, XY[1][1]); ZZ[1] = ffma2s(r1.x, W1, ZZ[1]);
                        XY[0][2] = ffma2s(W2.x, g01, XY[0][2]); XY[1][2] = ffma2s(W2.y, g01, XY[1][2]); ZZ[2] = ffma2s(r1.x, W2, ZZ[2]);
                        if (ox == 0) { gown[rr - 1][0] = r0.z; gown[rr - 1][1] = r0.w; gown[rr - 1][2] = r1.x; }
                    }
                }
            }
            // ---- direct + position terms ----
            if (s >= zs && s < ze) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    if (!act[j] || (j == 0 ? nz1 : nz2) == 0) continue;
                    const int lc = lc0 + j * BW;
                    const float g0 = gown[j][0], g1 = gown[j][1], g2 = gown[j][2];
                    float px = xf + Us[lc] * c.in_scale, py = (float)(y0 + j) + Us[CS + lc] * c.in_scale,
                          pz = (float)s + Us[2 * CS + lc] * c.in_scale;
                    const float mx = irs_inside(px, d.W) * c.in_scale, my = irs_inside(py, d.H) * c.in_scale,
                                mz = irs_inside(pz, d.D) * c.in_scale;
                    px = irs_clampf(px, 0.f, xmax); py = irs_clampf(py, 0.f, ymax); pz = irs_clampf(pz, 0.f, zmax);
                    const float fx0 = floorf(px), fy0 = floorf(py), fz0 = floorf(pz);
                    const float fx = px - fx0, fy = py - fy0, fz = pz - fz0;
                    const int ix = (int)fx0, iy = (int)fy0, iz = (int)fz0;
                    const int s0 = (it + 1 + (iz - s)) & (TMA_NS - 1), s1 = (s0 + 1) & (TMA_NS - 1);
                    const int i000 = s0 * SS + (iy - (c.y0t - 1)) * BW + (ix - (c.x0t - TMA_XO));
                    float jx, jy, jz;
                    ring_interp_grad_dot<BW>(c.U, CS, i000, (s1 - s0) * SS, g0, g1, g2, fx, fy, fz, jx, jy, jz);
                    XY[j][1].x += g0 + mx * jx;
                    XY[j][1].y += g1 + my * jy;
                    if (j == 0) ZZ[1].x += g2 + mz * jz; else ZZ[1].y += g2 + mz * jz;
                }
            }
        }
        // ---- target plane s-1 is complete ----
        if (s - 1 >= zs && s - 1 < ze) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                if (act[j]) {
                    const int o = gi + j * d.W;
                    c.g[o] = XY[j][0].x * c.out_scale;
                    c.g[Vi + o] = XY[j][0].y * c.out_scale;
                    c.g[2 * Vi + o] = (j == 0 ? ZZ[0].x : ZZ[0].y) * c.out_scale;
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) { XY[j][0] = XY[j][1]; XY[j][1] = XY[j][2]; XY[j][2] = make_float2(0.f, 0.f); }
        ZZ[0] = ZZ[1]; ZZ[1] = ZZ[2]; ZZ[2] = make_float2(0.f, 0.f);
        gi += HW;
        __syncthreads();
        if (tid == 0) {
            if (it + 4 < n_u) {
                irs_mbar_expect_tx(&c.bar_u[it & 3], B2_BYTES);
                irs_tma_load_plane(c.U + (it & 3) * SS, c.tmap_u, &c.bar_u[it & 3], c.x0t - TMA_XO, c.y0t - 1, zs + 2 + it,
                                   3 * c.chain);
            }
            if (it + 1 + BWD_NG < n_g) {
                irs_mbar_expect_tx(&c.bar_g[BP], B2_BYTES);
                irs_tma_load_plane(c.G + BP * SS, c.tmap_g, &c.bar_g[BP], c.x0t - TMA_XO, c.y0t - 1, zs + 3 + it, 3 * c.chain);
            }
        }
    }
}

__global__ void __launch_bounds__(TILE_T, 2)
svf_step_bwd_tma2_kernel(const __grid_constant__ CUtensorMap tmap_u, const __grid_constant__ CUtensorMap tmap_g,
                         const float* __restrict__ in, float in_scale, const float* __restrict__ gp_all,
                         float* __restrict__ g_all, const float* __restrict__ maxabs, int radius_max, float out_scale,
                         int seg_len, IrsDims d, IrsCells cm) {
    extern __shared__ __align__(128) float smem[];
    irs_pdl_wait();
    irs_pdl_launch_dependents();
    const int R = svf_gather_radius(__ldg(maxabs));
    const long long V = d.V();
    const size_t off = (size_t)blockIdx.y * 3 * V;
    const int tiles_x = (d.W + TILE_X - 1) / TILE_X, tiles_y = (d.H + B2_TY - 1) / B2_TY;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int x0t = bx * TILE_X, y0t = by * B2_TY, zs = bz * seg_len, ze = min(zs + seg_len, d.D);
    const int Rl = svf_local_radius(R, radius_max, cm, blockIdx.y, x0t, y0t, B2_TY, zs, ze);
    if (Rl == 1 && Rl <= radius_max) {
        BwdTmaCtx c;
        c.tmap_u = &tmap_u; c.tmap_g = &tmap_g;
        c.U = smem;
        c.G = smem + TMA_NS * B2_SS;
        c.REC = smem + (TMA_NS + BWD_NG) * B2_SS;
        c.bar_u = reinterpret_cast<uint64_t*>(c.REC + 2 * B2_NR * REC_F);
        c.bar_g = c.bar_u + TMA_NS;
        c.row_nz = reinterpret_cast<int*>(c.bar_g + BWD_NG);
        c.in_scale = in_scale; c.out_scale = out_scale; c.d = d;
        c.x0t = x0t; c.y0t = y0t; c.zs = zs; c.ze = ze; c.chain = blockIdx.y;
        c.g = g_all + off;
        svf_bwd_tma2_body(c);
    } else {   // the 32 x 8 fallbacks, once per half tile
        svf_bwd_tile_dispatch_cold(R, in + off, in_scale, gp_all + off, g_all + off, radius_max, out_scale, d, x0t, y0t, zs, ze,
                                   smem);
        __syncthreads();
        if (y0t + TILE_Y < d.H)
            svf_bwd_tile_dispatch_cold(R, in + off, in_scale, gp_all + off, g_all + off, radius_max, out_scale, d, x0t,
                                       y0t + TILE_Y, zs, ze, smem);
    }
}

constexpr size_t svf_bwd_tile_smem(int R) {
    return sizeof(float) * (size_t)(3 * (2 * R + 1) + 3) * (TILE_X + 2 * R) * (TILE_Y + 2 * R);
}
constexpr size_t svf_fwd_tile_smem(int R) {
    return sizeof(float) * (size_t)(3 * (2 * R + 1)) * 64 * (TILE_Y + 2 * R);
}

// z-segment length: the (tiles x segments x chains) CTAs should fill whole waves of the 148 SMs, while each segment
// pays `halo` extra plane-iterations.  Picks the segment count with the lowest modelled time.
// `dynamic`: the TMA kernels' CTAs differ in cost (zero-gradient rows are skipped), so more CTAs than resident slots let
// the hardware scheduler even the SMs out; measured at 128^3, one chain: 10 (adjoint) / 8 (forward) planes beat 15.
static int svf_seg_len(IrsDims d, int C, int slots, int halo, const char* env_name = "IRS_SVF_SEG", bool dynamic = false,
                       int tile_y = TILE_Y) {
    if (const char* e = getenv(env_name)) {   // test hook: forces segment boundaries; read at every launch
        const int v = atoi(e);
        if (v >= 1) return v < d.D ? v : d.D;
    }
    const long long tiles = (long long)((d.W + TILE_X - 1) / TILE_X) * ((d.H + tile_y - 1) / tile_y) * C;
    int best_len = d.D;
    double best_cost = 1e300;
    for (int nseg = 1; nseg <= d.D; ++nseg) {
        const int len = (d.D + nseg - 1) / nseg;
        if (len > 32 && len < d.D) continue;   // measured: long segments lose more to load imbalance than they save in halo
        if (len > 32 && nseg == 1 && d.D > 32) continue;
        if (len < 4 && nseg > 1) break;
        const int nseg_eff = (d.D + len - 1) / len;
        const long long ctas = tiles * nseg_eff;
        const long long waves = (ctas + slots - 1) / slots;
        const double fill = (double)ctas / slots;
        const double cost = dynamic ? ((fill > 1.0 ? fill : 1.0) + 0.35) * (len + halo) : (double)waves * (len + halo);
        if (cost < best_cost - 1e-9) { best_cost = cost; best_len = len; }
    }
    return best_len;
}

__global__ void __launch_bounds__(256)
svf_outputs_kernel(const float* __restrict__ u_all, const float* __restrict__ lin_x, const float* __restrict__ lin_y,
                   const float* __restrict__ lin_z, float* __restrict__ T, float* __restrict__ disp, IrsDims d) {
    const long long V = d.V();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const int c = blockIdx.y;
    const float* u = u_all + (size_t)c * 3 * V;
    const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), z = (int)(i / ((long long)d.W * d.H));
    const float ux = u[i], uy = u[V + i], uz = u[2 * V + i];
    if (disp != nullptr) {
        float* o = disp + (size_t)c * 3 * V;
        o[i] = ux; o[V + i] = uy; o[2 * V + i] = uz;
    }
    if (T != nullptr) {
        // reference utils/util.py:418-429: channel idx scaled by 2/(shape[2+idx]-1) (sic), identity = fp32 linspace
        float* o = T + (size_t)c * 3 * V;
        o[i] = lin_x[x] + ux * (2.0f / (float)(d.D - 1));
        o[V + i] = lin_y[y] + uy * (2.0f / (float)(d.H - 1));
        o[2 * V + i] = lin_z[z] + uz * (2.0f / (float)(d.W - 1));
    }
}

// Launch configuration that depends on the device: the opt-in shared-memory size is a per-device function attribute and
// the resident-CTA counts come from that device's occupancy calculator.  A process that drives several GPUs (one sampler per
// device) must not reuse the first device's state, so everything is cached PER DEVICE behind a mutex.
struct SvfDeviceState {
    bool fwd_tma_ready = false, bwd_tile_ready = false, bwd_tma2_ready = false;
    int slots_fwd_tma = 0, slots_fwd_tile = 0, slots_bwd_tile = 0, slots_bwd_tma = 0;
};
constexpr int kMaxDevices = 64;
SvfDeviceState g_svf_dev[kMaxDevices];
std::mutex g_svf_mu;
inline SvfDeviceState& svf_device_state() {
    int dev = 0;
    cudaGetDevice(&dev);
    return g_svf_dev[(dev % kMaxDevices + kMaxDevices) % kMaxDevices];
}

template <typename K>
static int resident_ctas(K kernel, size_t smem) {
    int per_sm = 0, sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TILE_T, smem) != cudaSuccess || per_sm < 1) per_sm = 2;
    return per_sm * sms;
}

}  // namespace

static size_t zmax(size_t a, size_t b) { return a > b ? a : b; }

// upper bound on the forward grid (x dimension) for a volume: segments are never shorter than 4 planes
size_t irs_svf_fwd_max_blocks(IrsDims d) {
    return (size_t)((d.W + TILE_X - 1) / TILE_X) * ((d.H + TILE_Y - 1) / TILE_Y) * ((d.D + 3) / 4);
}

int irs_launch_svf_fwd(const float* v, float* hist, float* maxabs, int n_steps, int C, IrsDims d, cudaStream_t st,
                       double* energy, long long energy_stride, double* partials, unsigned int* counters,
                       int* energy_done) {
    if (energy_done) *energy_done = 0;
    const size_t F = (size_t)C * 3 * d.V();
    cudaError_t e = cudaMemsetAsync(maxabs, 0, sizeof(float) * n_steps, st);   // the cell maps are written, not accumulated
    if (e != cudaSuccess) return (int)e;
    const float scale0 = 1.0f / (float)(1 << n_steps);
    // Cell map of the input of step k (= the field the adjoint of step k gathers from).  Only the last four steps can reach one
    // voxel for |v| < 16 voxels (|u_k| <= |v| / 2^(n-k)); earlier steps keep the step-wide radius.  The kernel exits at once
    // unless max |u_k| >= 1, and with programmatic dependent launch it is invisible in graph replay.
    // one launch behind the whole forward pass (the maps are read by the adjoint only)
    auto launch_cells = [&]() -> cudaError_t {
        const int k_first = n_steps > 4 ? n_steps - 4 : 1;
        if (k_first >= n_steps) return cudaSuccess;
        IrsCells cm = make_cells(maxabs, n_steps, k_first, C, d);
        dim3 grid((unsigned)(cm.nx * cm.ny * cm.nz), C, n_steps - k_first);
        return irs_launch_pdl(svf_cells_kernel, grid, dim3(256), 0, st, v, (const float*)hist, scale0, maxabs, n_steps, k_first,
                              (long long)F, C, d);
    };
    constexpr int RF = 2;
    const int tiles = ((d.W + TILE_X - 1) / TILE_X) * ((d.H + TILE_Y - 1) / TILE_Y);
    const bool tma = irs_tma_field_ok(v, d.W) && irs_tma_field_ok(hist, d.W) && (F % 4) == 0;
    if (tma) {
        const size_t smem = zmax(svf_fwd_tma_smem(), svf_fwd_tile_smem_compact(RF));
        auto* const kern = svf_step_fwd_tma_kernel<false>;
        auto* const kern_e = svf_step_fwd_tma_kernel<true>;
        int slots = 0;
        {
            std::lock_guard<std::mutex> lock(g_svf_mu);
            SvfDeviceState& ds = svf_device_state();
            if (!ds.fwd_tma_ready) {
                e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return (int)e;
                e = cudaFuncSetAttribute(kern_e, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return (int)e;
                ds.slots_fwd_tma = resident_ctas(kern, smem);
                ds.fwd_tma_ready = true;
            }
            slots = ds.slots_fwd_tma;
        }
        const int seg_len = svf_seg_len(d, C, slots, 3, "IRS_SVF_SEG_FWD", true);
        dim3 tgrid(tiles * ((d.D + seg_len - 1) / seg_len), C);
        // the first step can reduce the regulariser energy of v on the way (its ring holds every neighbour)
        const bool with_energy = energy != nullptr && partials != nullptr && counters != nullptr &&
                                 (size_t)tgrid.x <= irs_svf_fwd_max_blocks(d);
        for (int k = 0; k < n_steps; ++k) {
            const float* in = (k == 0) ? v : hist + (size_t)(k - 1) * F;
            CUtensorMap map;
            if (irs_tma_encode_field(&map, in, 3 * C, d.D, d.H, d.W, FWD_BW, TMA_EY) != 0) return IRS_ERR_UNSUPPORTED;
            const bool en = with_energy && k == 0;
            IrsEnergyOut eo{en ? energy : nullptr, energy_stride, partials, counters};
            e = irs_launch_pdl(en ? kern_e : kern, tgrid, dim3(TILE_T), smem, st, map, in, k == 0 ? scale0 : 1.0f,
                               hist + (size_t)k * F, k == 0 ? nullptr : maxabs + k - 1, maxabs + k, seg_len, d, eo);
            if (e != cudaSuccess) return (int)e;
        }
        e = launch_cells();
        if (e != cudaSuccess) return (int)e;
        if (with_energy && energy_done) *energy_done = 1;
        return (int)cudaGetLastError();
    }
    int slots = 0;
    {
        std::lock_guard<std::mutex> lock(g_svf_mu);
        SvfDeviceState& ds = svf_device_state();
        if (ds.slots_fwd_tile == 0) {
            e = cudaFuncSetAttribute(svf_step_fwd_tile_kernel<RF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)svf_fwd_tile_smem(RF));
            if (e != cudaSuccess) return (int)e;
            ds.slots_fwd_tile = resident_ctas(svf_step_fwd_tile_kernel<RF>, svf_fwd_tile_smem(RF));
        }
        slots = ds.slots_fwd_tile;
    }
    const int seg_len = svf_seg_len(d, C, slots, 2 * RF + 2);
    dim3 tgrid(tiles * ((d.D + seg_len - 1) / seg_len), C);
    for (int k = 0; k < n_steps; ++k) {
        const float* in = (k == 0) ? v : hist + (size_t)(k - 1) * F;
        e = irs_launch_pdl(svf_step_fwd_tile_kernel<RF>, tgrid, dim3(TILE_T), svf_fwd_tile_smem(RF), st, in,
                           k == 0 ? scale0 : 1.0f, hist + (size_t)k * F, maxabs + k, seg_len, d);
        if (e != cudaSuccess) return (int)e;
    }
    e = launch_cells();
    if (e != cudaSuccess) return (int)e;
    return (int)cudaGetLastError();
}

int irs_launch_svf_bwd(const float* v, const float* hist, const float* maxabs, float* g_u, float* g_work, float* g_v,
                       int n_steps, int gather_radius_max, int C, IrsDims d, cudaStream_t st) {
    const size_t F = (size_t)C * 3 * d.V();
    const float scale0 = 1.0f / (float)(1 << n_steps);
    const size_t smem = svf_bwd_tile_smem(2);
    const long long vblocks = (d.V() + 255) / 256;
    dim3 vgrid((unsigned)(vblocks < 1184 ? vblocks : 1184), 1);   // persistent: see svf_step_bwd_scatter_kernel
    const bool tma = irs_tma_field_ok(v, d.W) && irs_tma_field_ok(hist, d.W) && irs_tma_field_ok(g_u, d.W) &&
                     irs_tma_field_ok(g_work, d.W) && (F % 4) == 0;
    const size_t smem_tma = zmax(svf_bwd_tma2_smem(), smem);
    int slots = 0, slots_tma = 0;
    {
        std::lock_guard<std::mutex> lock(g_svf_mu);
        SvfDeviceState& ds = svf_device_state();
        if (!ds.bwd_tile_ready) {
            cudaError_t e = cudaFuncSetAttribute(svf_step_bwd_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return (int)e;
            ds.slots_bwd_tile = resident_ctas(svf_step_bwd_tile_kernel, smem);
            ds.bwd_tile_ready = true;
        }
        if (tma && !ds.bwd_tma2_ready) {
            cudaError_t e = cudaFuncSetAttribute(svf_step_bwd_tma2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tma);
            if (e != cudaSuccess) return (int)e;
            ds.slots_bwd_tma = resident_ctas(svf_step_bwd_tma2_kernel, smem_tma);
            ds.bwd_tma2_ready = true;
        }
        slots = ds.slots_bwd_tile;
        slots_tma = ds.slots_bwd_tma;
    }
    const int tile_y = tma ? B2_TY : TILE_Y;
    const int seg_len = tma ? svf_seg_len(d, C, slots_tma, 4, "IRS_SVF_SEG_BWD", true, tile_y) : svf_seg_len(d, C, slots, 6);
    const int tiles = ((d.W + TILE_X - 1) / TILE_X) * ((d.H + tile_y - 1) / tile_y);
    dim3 tgrid(tiles * ((d.D + seg_len - 1) / seg_len), C);
    // ping-pong between g_work and the caller's g_u buffer (g_u is only read by the first adjoint step)
    const float* gp = g_u;
    cudaError_t le = cudaSuccess;
    for (int k = n_steps - 1; k >= 0; --k) {
        const float* in = (k == 0) ? v : hist + (size_t)(k - 1) * F;
        float* out = (k == 0) ? g_v : (((n_steps - 1 - k) & 1) ? g_u : g_work);
        const float in_scale = (k == 0) ? scale0 : 1.0f;
        // Only the last four steps can reach displacements beyond the gather limit for |v| < 32 voxels (|u_k| <= |v| /
        // 2^(n-k)); they get the early-exit scatter companion.  Earlier steps gather with whatever radius their max |u_k|
        // asks for (exact; slow only for absurd fields), which saves eight empty launches per transition.
        // the forward pass left the cell map of u_k behind the n_steps global maxima for the last four steps (read-only here)
        IrsCells cm = make_cells(const_cast<float*>(maxabs), n_steps, k, C, d);
        if (k < n_steps - 4 || k == 0) cm.p = nullptr;
        const bool companion = k >= n_steps - 4;
        const int radius_max_k = companion ? gather_radius_max : 0x7fffffff;
        if (tma) {
            CUtensorMap map_u, map_g;
            if (irs_tma_encode_field(&map_u, in, 3 * C, d.D, d.H, d.W, BWD_BW, B2_EY) != 0 ||
                irs_tma_encode_field(&map_g, gp, 3 * C, d.D, d.H, d.W, BWD_BW, B2_EY) != 0)
                return IRS_ERR_UNSUPPORTED;
            le = irs_launch_pdl(svf_step_bwd_tma2_kernel, tgrid, dim3(TILE_T), smem_tma, st, map_u, map_g, in, in_scale, gp,
                                out, maxabs + k, radius_max_k, in_scale, seg_len, d, cm);
        } else {
            le = irs_launch_pdl(svf_step_bwd_tile_kernel, tgrid, dim3(TILE_T), smem, st, in, in_scale, gp, out, maxabs + k,
                                radius_max_k, in_scale, seg_len, d, cm);
        }
        if (le != cudaSuccess) return (int)le;
        if (companion) {
            le = irs_launch_pdl(svf_step_bwd_scatter_kernel, vgrid, dim3(256), 0, st, in, in_scale, gp, (float*)out, maxabs + k,
                                gather_radius_max, in_scale, C, d);
            if (le != cudaSuccess) return (int)le;
        }
        gp = out;
    }
    return (int)cudaGetLastError();
}

// n_steps global maxima followed by n_steps cell maps (C x cells of 32 x 8 x 8 voxels)
extern "C" size_t irs_svf_maxabs_floats(int C, int D, int H, int W, int n_steps) {
    if (C < 1 || D < 1 || H < 1 || W < 1 || n_steps < 1) return 0;
    return (size_t)n_steps * (1 + (size_t)C * irs_cells_per_chain(IrsDims{D, H, W}));
}

extern "C" size_t irs_svf_hist_floats(int C, int D, int H, int W, int n_steps) {
    return (size_t)n_steps * C * 3 * D * H * W;
}

extern "C" int irs_svf_exp_fwd(const float* v, float* hist, float* maxabs, int n_steps, int C, int D, int H, int W,
                               void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    IRS_CHECK_CUBE(D, H, W);
    if (!v || !hist || !maxabs || n_steps < 1 || n_steps > IRS_MAX_SVF_STEPS) return IRS_ERR_BAD_ARG;
    return irs_launch_svf_fwd(v, hist, maxabs, n_steps, C, IrsDims{D, H, W}, (cudaStream_t)stream, nullptr, 0, nullptr, nullptr,
                              nullptr);
}

extern "C" int irs_svf_outputs(const float* u, const float* lin_x, const float* lin_y, const float* lin_z, float* T,
                               float* disp, int C, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    IRS_CHECK_CUBE(D, H, W);
    if (!u || (T && (!lin_x || !lin_y || !lin_z))) return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    dim3 grid((unsigned)((d.V() + 255) / 256), C);
    svf_outputs_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(u, lin_x, lin_y, lin_z, T, disp, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_svf_exp_bwd(const float* v, const float* hist, const float* maxabs, float* g_u, float* g_work,
                               float* g_v, int n_steps, int gather_radius_max, int C, int D, int H, int W,
                               void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    IRS_CHECK_CUBE(D, H, W);
    if (!v || !hist || !maxabs || !g_u || !g_work || !g_v || n_steps < 1 || n_steps > IRS_MAX_SVF_STEPS)
        return IRS_ERR_BAD_ARG;
    if (gather_radius_max < 0) return IRS_ERR_BAD_ARG;
    return irs_launch_svf_bwd(v, hist, maxabs, g_u, g_work, g_v, n_steps, gather_radius_max, C, IrsDims{D, H, W},
                              (cudaStream_t)stream);
}
