// irs_data.cu -- data term: LCC normalisation as separable box filters over shared-memory tiles with halos, its adjoint,
// the Gaussian-mixture log-density with warp-shuffle reductions, virtual decimation.
// (reference model/loss.py:87-114, utils/util.py:330-347,446-485, trainer/trainer.py:68-77,316-327)
#include <type_traits>

#include "irs_kernels.cuh"

namespace {

constexpr int TX = 32, TY = 8;  // in-plane tile of the box filters; 256 threads = TX x TY

enum { BOX_FWD_MEAN = 0, BOX_FWD_VAR = 1, BOX_BWD_VAR = 2, BOX_BWD_MEAN = 3, BOX_BWD_MEAN_WARP = 4 };

// weight of input offset o for output position j in the ADJOINT of a replicate-padded box of half width S:
// the out-of-range window positions of a border voxel were clamped onto it in the forward pass (fold)
__device__ __forceinline__ float adj_weight(int j, int o, int n, int S) {
    float w = 1.f;
    if (j == 0 && o >= 0) w += (float)(S - o);
    if (j == n - 1 && o <= 0) w += (float)(S + o);
    return w;
}

// One 3-D box filter (forward: replicate padding; backward: its adjoint) with a fused pre-operation on the loaded values
// and a fused epilogue:
//   FWD_MEAN : in0 = I                       -> out0 = a = I - box(I)/k^3
//   FWD_VAR  : in0 = a (pre: a^2), in1 = zF  -> out0 = rs = 1/sqrt(box/k^3 + 1e-10), out1 = z = zF - a rs  (zF null: a rs)
//   BWD_VAR  : in0 = g, in1 = a, in2 = rs (pre: -g a rs^3 / 2) -> out0 = ga = g rs + 2 a adjbox/k^3        (g = sign * in0)
//   BWD_MEAN : in0 = ga                      -> out0 = ga - adjbox/k^3
//   BWD_MEAN_WARP : the same value g, then out0 (C,3,V) = g * out0 in place: out0 holds the warp's spatial gradient
//              (irs_launch_warp_vox_fwd), the product is dL/du -- the warp adjoint as an epilogue
// Plane-marching form: a CTA owns a 32 x 8 column of voxels and walks along a z segment.  Per plane: tile + halo S in
// x / y goes through registers into a double-buffered shared-memory plane (pre-operation applied), x pass -> shared
// memory, y pass -> one register per thread, and the z pass is a ring of 2S+1 registers; the next plane's global loads
// are in flight while this plane is filtered.  (Round-1 history: a 32 x 8 x 8 tile with a z halo inside the tile and
// three shared-memory passes ran 47 / 48 us for the forward / adjoint pair at 128^3; this form 39 / 42 us.)
template <int MODE, int S>
__global__ void __launch_bounds__(256)
box_march_kernel(const float* __restrict__ in0, const float* __restrict__ in1, const float* __restrict__ in2, float sign,
                 float* __restrict__ out0, float* __restrict__ out1, int seg_len, IrsDims d) {
    constexpr int EX = TX + 2 * S, EY = TY + 2 * S, NP = EX * EY, NE = (NP + 255) / 256, NT = 2 * S + 1;
    constexpr bool BWD = (MODE == BOX_BWD_VAR || MODE == BOX_BWD_MEAN || MODE == BOX_BWD_MEAN_WARP);
    __shared__ float P[2][NP];        // plane tile + halo (pre-operation applied), double-buffered
    __shared__ float X[EY * TX];      // x-pass result

    const int V = (int)d.V(), HW = d.H * d.W;
    const int c = blockIdx.y;
    const int tiles_x = (d.W + TX - 1) / TX, tiles_y = (d.H + TY - 1) / TY;
    const int bx = blockIdx.x % tiles_x, by = (blockIdx.x / tiles_x) % tiles_y, bz = blockIdx.x / (tiles_x * tiles_y);
    const int x0 = bx * TX, y0 = by * TY, zs = bz * seg_len, ze = min(zs + seg_len, d.D);
    const size_t off = (size_t)c * V;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
    const int gx = x0 + lx, gy = y0 + ly;
    const bool active = gx < d.W && gy < d.H;
    const float* p0 = in0 + off;
    const float* p1 = in1 ? in1 + off : nullptr;
    const float* p2 = in2 ? in2 + off : nullptr;

    // the plane elements this thread stages: offsets inside a (H, W) plane (forward: clamped = replicate padding;
    // adjoint: -1 outside the volume = zero) and inside the shared-memory plane
    int pofs[NE], sofs[NE];
#pragma unroll
    for (int k = 0; k < NE; ++k) {
        const int e = threadIdx.x + k * 256;
        const int ey = e / EX, ex = e - ey * EX;
        const int ax = x0 - S + ex, ay = y0 - S + ey;
        sofs[k] = e < NP ? e : -1;
        if (BWD) pofs[k] = (e < NP && ax >= 0 && ax < d.W && ay >= 0 && ay < d.H) ? ay * d.W + ax : -1;
        else pofs[k] = irs_clampi(ay, 0, d.H - 1) * d.W + irs_clampi(ax, 0, d.W - 1);
    }
    float raw[MODE == BOX_BWD_VAR ? 3 : 1][NE];
    auto fetch = [&](int pz) {   // global loads of plane pz into registers (values finished in stage())
        int zofs;
        bool zin = true;
        if (BWD) { zin = pz >= 0 && pz < d.D; zofs = pz * HW; }
        else zofs = irs_clampi(pz, 0, d.D - 1) * HW;
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            const bool ok = sofs[k] >= 0 && zin && pofs[k] >= 0;
            const int gi = zofs + pofs[k];
            raw[0][k] = ok ? __ldg(p0 + gi) : 0.f;
            if (MODE == BOX_BWD_VAR) {
                raw[1][k] = ok ? __ldg(p1 + gi) : 0.f;
                raw[2][k] = ok ? __ldg(p2 + gi) : 0.f;
            }
        }
    };
    auto stage = [&](int buf) {  // pre-operation + store into the shared-memory plane
#pragma unroll
        for (int k = 0; k < NE; ++k) {
            if (sofs[k] < 0) continue;
            float v = raw[0][k];
            if (MODE == BOX_FWD_VAR) v = v * v;
            if (MODE == BOX_BWD_VAR) { const float r = raw[2][k]; v = -0.5f * (sign * v) * raw[1][k] * r * r * r; }
            P[buf][sofs[k]] = v;
        }
    };

    // adjoint: the fold weights differ from 1 only for outputs on a face of the volume
    const bool fold_x = BWD && (x0 == 0 || x0 + TX >= d.W), fold_y = BWD && (y0 == 0 || y0 + TY >= d.H);
    const float inv_k3 = 1.0f / (float)((2 * S + 1) * (2 * S + 1) * (2 * S + 1));

    float ring[NT];   // y-pass results of the last 2S+1 planes (ring[NT-1] = newest)
#pragma unroll
    for (int i = 0; i < NT; ++i) ring[i] = 0.f;

    const int p_first = zs - S, p_last = ze - 1 + S;
    fetch(p_first);
    stage(0);
    __syncthreads();
    for (int p = p_first, it = 0; p <= p_last; ++p, ++it) {
        const int buf = it & 1;
        if (p < p_last) fetch(p + 1);   // in flight while this plane is filtered
        // ---- x pass: X[row][x] = sum_o w P[row][x + S + o], rows ly and ly + 8 ----
#pragma unroll
        for (int r = 0; r < (EY + 7) / 8; ++r) {
            const int row = ly + 8 * r;
            if (row < EY) {
                const float* a = &P[buf][row * EX + lx + S];
                float acc = 0.f;
                if (fold_x) {
#pragma unroll
                    for (int o = -S; o <= S; ++o) acc += adj_weight(gx, o, d.W, S) * a[o];
                } else {
#pragma unroll
                    for (int o = -S; o <= S; ++o) acc += a[o];
                }
                X[row * TX + lx] = acc;
            }
        }
        __syncthreads();
        // ---- y pass into the register ring ----
#pragma unroll
        for (int i = 0; i < NT - 1; ++i) ring[i] = ring[i + 1];
        {
            const float* b = &X[(ly + S) * TX + lx];
            float acc = 0.f;
            if (fold_y) {
#pragma unroll
                for (int o = -S; o <= S; ++o) acc += adj_weight(gy, o, d.H, S) * b[o * TX];
            } else {
#pragma unroll
                for (int o = -S; o <= S; ++o) acc += b[o * TX];
            }
            ring[NT - 1] = acc;
        }
        // ---- z pass + epilogue for plane gz = p - S (its window p-2S .. p is in the ring) ----
        const int gz = p - S;
        if (active && gz >= zs && gz < ze) {
            float acc = 0.f;
            if (BWD && (gz == 0 || gz == d.D - 1)) {
#pragma unroll
                for (int o = -S; o <= S; ++o) acc += adj_weight(gz, o, d.D, S) * ring[o + S];
            } else {
#pragma unroll
                for (int o = -S; o <= S; ++o) acc += ring[o + S];
            }
            const float box = acc * inv_k3;
            const size_t gi = off + (size_t)gz * HW + gy * d.W + gx;
            if (MODE == BOX_FWD_MEAN) {
                out0[gi] = in0[gi] - box;
            } else if (MODE == BOX_FWD_VAR) {
                const float rs = 1.0f / sqrtf(box + 1e-10f);
                const float zn = in0[gi] * rs;
                if (out0 != nullptr) out0[gi] = rs;
                if (out1 != nullptr) out1[gi] = in1 != nullptr ? in1[gi - off] - zn : zn;
            } else if (MODE == BOX_BWD_VAR) {
                out0[gi] = sign * in0[gi] * in2[gi] + 2.0f * in1[gi] * box;
            } else if (MODE == BOX_BWD_MEAN) {
                out0[gi] = in0[gi] - box;
            } else {
                const float g = in0[gi] - box;
                float* w = out0 + 3 * off + (size_t)gz * HW + gy * d.W + gx;
                w[0] = g * w[0]; w[V] = g * w[V]; w[2 * (size_t)V] = g * w[2 * (size_t)V];
            }
        }
        if (p < p_last) stage(buf ^ 1);
        __syncthreads();
    }
}

static int box_seg_len(IrsDims d, int C) {
    // enough CTAs for ~2 waves of the 148 x 8 resident slots, segments no shorter than 8 planes (halo 2S per segment)
    const long long tiles = (long long)((d.W + TX - 1) / TX) * ((d.H + TY - 1) / TY) * C;
    int len = d.D;
    while (len > 8 && tiles * ((d.D + len - 1) / len) < 2 * 1184) len = (len + 1) / 2;
    return len < 8 ? (d.D < 8 ? d.D : 8) : len;
}

template <int MODE, int S>
int launch_box_s(const float* in0, const float* in1, const float* in2, float sign, float* out0, float* out1, int C,
                 IrsDims d, cudaStream_t st) {
    const int seg_len = box_seg_len(d, C);
    const int tiles = ((d.W + TX - 1) / TX) * ((d.H + TY - 1) / TY) * ((d.D + seg_len - 1) / seg_len);
    dim3 grid(tiles, C);
    box_march_kernel<MODE, S><<<grid, 256, 0, st>>>(in0, in1, in2, sign, out0, out1, seg_len, d);
    return (int)cudaGetLastError();
}

template <int MODE>
int launch_box(const float* in0, const float* in1, const float* in2, float sign, float* out0, float* out1, int S, int C,
               IrsDims d, cudaStream_t st) {
    switch (S) {
        case 1: return launch_box_s<MODE, 1>(in0, in1, in2, sign, out0, out1, C, d, st);
        case 2: return launch_box_s<MODE, 2>(in0, in1, in2, sign, out0, out1, C, d, st);
        case 3: return launch_box_s<MODE, 3>(in0, in1, in2, sign, out0, out1, C, d, st);
        default: return IRS_ERR_UNSUPPORTED;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// mixture statistics of one chain with the CURRENT parameters, then (last block) virtual decimation factor + Adam step
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float masked_vd_residual(const IrsGmm& g, const float* __restrict__ z,
                                                    const unsigned char* __restrict__ mask, long long i) {
    return mask[i] ? irs_gmm_vd_residual(g, __ldg(z + i)) : 0.f;
}

// The scalar tail of a chain's mixture step, run by ONE WARP (call with the first 32 threads of the CTA that holds the reduced
// sums): Adam with one lane per parameter, the table with one lane per component.  Bit-identical to the serial composition
// irs_gmm_adam_step + irs_gmm_table (irs_hyper.cuh) -- this is the critical path between two chains, and as a loop on one thread
// it cost 5-8 us of expf / logf / fp64 latency.
__device__ __forceinline__ void gmm_finalize_warp(double* __restrict__ hyper, const IrsHyperCfg& cfg, const double* total,
                                                  double alpha32, bool frozen, float* __restrict__ table_out,
                                                  double* __restrict__ stats_row) {
    const int lane = threadIdx.x & 31;
    if (!frozen) {
        IrsAdamCtx ctx;
        irs_gmm_adam_context(hyper, cfg, total, ctx);
        __syncwarp();
        if (lane < 2 * cfg.K) irs_gmm_adam_param(hyper, cfg, total, alpha32, ctx, lane);
        __syncwarp();
        if (lane == 0) irs_gmm_adam_advance(hyper, cfg);
        __syncwarp();
    }
    float logpi[IRS_MAX_K];
    irs_log_proportions(hyper + IRS_HYPER_LOGITS, cfg.K, logpi);
    if (lane < IRS_MAX_K) {   // irs_gmm_table, one lane per component
        const float lsk = lane < cfg.K ? (float)hyper[IRS_HYPER_LOG_STD + lane] : 0.f;
        table_out[lane] = lane < cfg.K ? logpi[lane] - lsk : -INFINITY;
        table_out[IRS_MAX_K + lane] = lane < cfg.K ? expf(-2.0f * lsk) : 0.f;
    }
    if (lane == 0) {
        stats_row[IRS_STAT_ALPHA] = alpha32;
        stats_row[IRS_STAT_NLL_PRE] = total[IRS_SUM_NLL];
    }
}

// mode 0: fused path (parameters from `hyper`, Adam step + table/alpha outputs; alpha_fixed != null reuses a stored
//         factor instead of recomputing it -- the 25 warm-up steps of trainer.py:544-547)
// mode 1: op-level VD factor only (mixture passed by value)
// mode 2: VD factor with the parameters in `hyper`, no Adam step
template <int MODE>
__global__ void __launch_bounds__(256)
gmm_stats_kernel(const float* __restrict__ z, const unsigned char* __restrict__ mask, double* __restrict__ hyper,
                 IrsGmm table_in, IrsHyperCfg cfg, double* __restrict__ partials, unsigned int* __restrict__ counter,
                 double* __restrict__ stats_row, float* __restrict__ table_out, double* __restrict__ alpha_out,
                 const double* __restrict__ alpha_fixed, IrsDims d) {
    __shared__ IrsGmm g;
    __shared__ double sh[IRS_SUM_COUNT * 32];
    __shared__ double total[IRS_SUM_COUNT];
    if (threadIdx.x == 0) {
        if (MODE != 1) irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, cfg.K, g);
        else g = table_in;
    }
    __syncthreads();
    const IrsGmm gl = g;
    const long long V = d.V();
    const long long sy = d.W, sz = (long long)d.W * d.H;
    float acc[IRS_SUM_COUNT];
#pragma unroll
    for (int k = 0; k < IRS_SUM_COUNT; ++k) acc[k] = 0.f;

    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x) {
        if (!mask[i]) continue;  // off the mask r = 0: no contribution to any sum
        const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), zc = (int)(i / sz);
        const float zi = z[i];
        float rho[IRS_MAX_K], wp;
        const float lp = irs_gmm_eval(gl, zi, rho, wp);
        const float z2 = zi * zi, r = z2 * wp;
        acc[IRS_SUM_NLL] -= lp;
        acc[IRS_SUM_RR] += r * r;
        if (cfg.virtual_decimation) {
            if (zc < d.D - 1) acc[IRS_SUM_RD] += r * masked_vd_residual(gl, z, mask, i + sz);
            if (y < d.H - 1) acc[IRS_SUM_RH] += r * masked_vd_residual(gl, z, mask, i + sy);
            if (x < d.W - 1) acc[IRS_SUM_RW] += r * masked_vd_residual(gl, z, mask, i + 1);
        }
#pragma unroll
        for (int k = 0; k < IRS_MAX_K; ++k) if (k < gl.K) {
            acc[IRS_SUM_RHO + k] += rho[k];
            acc[IRS_SUM_Q + k] += rho[k] * z2 * gl.prec[k];
        }
    }
    double blk[IRS_SUM_COUNT];
    irs_block_sum<IRS_SUM_COUNT>(acc, blk, sh);
    if (!irs_grid_sum<IRS_SUM_COUNT>(blk, partials, counter, total)) return;
    if (threadIdx.x != 0) return;

    double n_mask = cfg.n_mask;
    if (!(n_mask > 0.0)) {  // responsibilities sum to one per masked voxel
        n_mask = 0.0;
        for (int k = 0; k < cfg.K; ++k) n_mask += total[IRS_SUM_RHO + k];
    }
    double alpha = cfg.virtual_decimation ? irs_vd_alpha(total, n_mask) : 1.0;
    if (MODE == 1) { *alpha_out = alpha; return; }
    if (MODE == 2) { stats_row[IRS_STAT_ALPHA] = irs_round_f32(alpha); return; }
    if (alpha_fixed != nullptr) alpha = *alpha_fixed;
    const double alpha32 = irs_round_f32(alpha);  // a fp32 scalar in the reference
    irs_gmm_adam_step(hyper, cfg, total, alpha32);
    IrsGmm up;
    irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, cfg.K, up);
    for (int k = 0; k < IRS_MAX_K; ++k) { table_out[k] = up.lw[k]; table_out[IRS_MAX_K + k] = up.prec[k]; }
    stats_row[IRS_STAT_ALPHA] = alpha32;
    stats_row[IRS_STAT_NLL_PRE] = total[IRS_SUM_NLL];
}

// ---- fused-step version of the above, split so that the mixture is evaluated once per voxel ----------------------------
// pass A: per masked voxel one mixture evaluation -> sums (NLL, sum r^2, rho_k, Q_k) and the VD residual r written out.
//         FINALIZE: no lag sums needed (virtual decimation off, or a stored factor is reused): the last block steps Adam.
template <bool FINALIZE>
__global__ void __launch_bounds__(256)
gmm_stats_a_kernel(const float* __restrict__ z, const unsigned char* __restrict__ mask, double* __restrict__ hyper,
                   IrsHyperCfg cfg, double* __restrict__ partials, unsigned int* __restrict__ counter,
                   float* __restrict__ r_out, double* __restrict__ totals_out, double* __restrict__ stats_row,
                   float* __restrict__ table_out, const double* __restrict__ alpha_fixed, int V) {
    __shared__ IrsGmm g;
    __shared__ double sh[IRS_SUM_COUNT * 32];
    __shared__ double total[IRS_SUM_COUNT];
    if (threadIdx.x == 0) irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, cfg.K, g);
    __syncthreads();
    const IrsGmm gl = g;
    float acc[IRS_SUM_COUNT];
#pragma unroll
    for (int k = 0; k < IRS_SUM_COUNT; ++k) acc[k] = 0.f;
    // one voxel; `on` = inside the mask.  Branch-free: the four voxels of a 128-bit load are evaluated side by side (the
    // loop is latency-bound on the exp / log chains), off-mask results are discarded by selects (adding 0 is exact).
    auto one = [&](auto kk_tag, float zi, bool on) {
        constexpr int KK = decltype(kk_tag)::value;
        float rho[KK], wp;
        const float lp = irs_gmm_eval_t<KK>(gl, zi, rho, wp);
        const float z2 = zi * zi, r = on ? z2 * wp : 0.f;
        acc[IRS_SUM_NLL] -= on ? lp : 0.f;
        acc[IRS_SUM_RR] += r * r;
#pragma unroll
        for (int k = 0; k < KK; ++k) if (k < gl.K) {
            acc[IRS_SUM_RHO + k] += on ? rho[k] : 0.f;
            acc[IRS_SUM_Q + k] += on ? rho[k] * z2 * gl.prec[k] : 0.f;
        }
        return r;
    };
    const bool vec = (V % 4 == 0) && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(mask) |
                                       reinterpret_cast<uintptr_t>(r_out)) & 15) == 0;
    auto sweep = [&](auto kk_tag) {
        if (vec) {   // 128-bit loads, four voxels per thread and iteration
            for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4; i < V; i += gridDim.x * blockDim.x * 4) {
                const uchar4 m4 = *reinterpret_cast<const uchar4*>(mask + i);
                float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m4.x | m4.y | m4.z | m4.w) {
                    const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + i));
                    r4.x = one(kk_tag, z4.x, m4.x != 0);
                    r4.y = one(kk_tag, z4.y, m4.y != 0);
                    r4.z = one(kk_tag, z4.z, m4.z != 0);
                    r4.w = one(kk_tag, z4.w, m4.w != 0);
                }
                if (!FINALIZE) *reinterpret_cast<float4*>(r_out + i) = r4;
            }
        } else {
            for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < V; i += gridDim.x * blockDim.x) {
                const float r = mask[i] ? one(kk_tag, z[i], true) : 0.f;
                if (!FINALIZE) r_out[i] = r;
            }
        }
    };
    if (gl.K <= 4) sweep(std::integral_constant<int, 4>{});
    else sweep(std::integral_constant<int, IRS_MAX_K>{});
    double blk[IRS_SUM_COUNT];
    irs_block_sum<IRS_SUM_COUNT>(acc, blk, sh);
    if (!irs_grid_sum<IRS_SUM_COUNT>(blk, partials, counter, total)) return;
    if (!FINALIZE) {
        if (threadIdx.x < IRS_SUM_COUNT) totals_out[threadIdx.x] = total[threadIdx.x];
        return;
    }
    if (threadIdx.x >= 32) return;
    const double alpha32 = irs_round_f32(alpha_fixed != nullptr ? *alpha_fixed : 1.0);
    gmm_finalize_warp(hyper, cfg, total, alpha32, false, table_out, stats_row);
}

// pass B: lag-1 products of r along D, H, W; the last block combines them with pass A's sums: VD factor, Adam step
__global__ void __launch_bounds__(256)
gmm_stats_b_kernel(const float* __restrict__ r, double* __restrict__ hyper, IrsHyperCfg cfg,
                   double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ totals,
                   double* __restrict__ stats_row, float* __restrict__ table_out, IrsDims d) {
    __shared__ double sh[3 * 32];
    __shared__ double total[3];
    const int V = (int)d.V(), sy = d.W, sz = d.W * d.H;
    float acc[3] = {0.f, 0.f, 0.f};
    if (d.W % 4 == 0 && (reinterpret_cast<uintptr_t>(r) & 15) == 0) {
        for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4; i < V; i += gridDim.x * blockDim.x * 4) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(r + i));
            if (a.x == 0.f && a.y == 0.f && a.z == 0.f && a.w == 0.f) continue;   // off the mask: no contribution
            const int x = i % d.W, y = (i / d.W) % d.H, zc = i / sz;
            if (zc < d.D - 1) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(r + i + sz));
                acc[0] += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
            }
            if (y < d.H - 1) {
                const float4 b = __ldg(reinterpret_cast<const float4*>(r + i + sy));
                acc[1] += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
            }
            const float nx = x + 4 < d.W ? __ldg(r + i + 4) : 0.f;
            acc[2] += a.x * a.y + a.y * a.z + a.z * a.w + a.w * nx;
        }
    } else {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < V; i += gridDim.x * blockDim.x) {
            const float ri = r[i];
            if (ri == 0.f) continue;   // off the mask (or an exactly zero residual): no contribution
            const int x = i % d.W, y = (i / d.W) % d.H, zc = i / sz;
            if (zc < d.D - 1) acc[0] += ri * __ldg(r + i + sz);
            if (y < d.H - 1) acc[1] += ri * __ldg(r + i + sy);
            if (x < d.W - 1) acc[2] += ri * __ldg(r + i + 1);
        }
    }
    double blk[3];
    irs_block_sum<3>(acc, blk, sh);
    if (!irs_grid_sum<3>(blk, partials, counter, total)) return;
    if (threadIdx.x >= 32) return;
    if (threadIdx.x == 0) { totals[IRS_SUM_RD] = total[0]; totals[IRS_SUM_RH] = total[1]; totals[IRS_SUM_RW] = total[2]; }
    __syncwarp();
    const double alpha32 = irs_round_f32(irs_vd_alpha(totals, cfg.n_mask));
    gmm_finalize_warp(hyper, cfg, totals, alpha32, false, table_out, stats_row);
}

// ---- all chains in ONE launch ----------------------------------------------------------------------------------------------
// The reference walks the chains in order and lets every chain step the SHARED mixture before the next one evaluates it
// (trainer/trainer.py:316-327): a chain of C dependent reductions.  As 2 C launches that is pure latency for small volumes
// (64 chains at 64^3: 24 % of the transition).  Here one persistent kernel (one CTA per SM, all resident) walks the chains:
// per chain every CTA reduces its share, the last CTA to arrive (irs_grid_sum) computes the virtual decimation factor, steps
// Adam, writes the chain's table and releases a ticket in global memory; the other CTAs wait for the ticket and go on with
// the next chain under the updated parameters.  The lag-1 products of virtual decimation are formed from residuals
// re-evaluated at the three forward neighbours (13 mixture evaluations per four voxels instead of 4) -- no residual field
// round trip, hence ONE grid-wide synchronisation per chain instead of two launches.
// SERIAL = false: the chains do not depend on each other (hyper_mode per_chain: a parameter block per chain; frozen: no
// Adam step at all) -- blockIdx.y = chain, no tickets.
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

constexpr int WALK_T = 512;        // threads per CTA
constexpr int WALK_PL = 4;         // planes per brick: 128 threads (= 512 voxels of one plane) per plane

// Sums of one chain over this CTA's share of the volume.  Vector path (W divides 512): the CTA walks over bricks of
// 4 planes x 512/W rows x W voxels, one float4 per thread; the residuals r of a brick go through shared memory, so the
// lag-1 products along x, y and z read their forward neighbour from there and only the brick's last row / last plane
// re-evaluates the mixture at the neighbour (1 + W/512 + 1/4 evaluations per voxel instead of 4).
template <int KK>
__device__ __noinline__ float gmm_halo4(const IrsGmm& gl, const float* __restrict__ z, const unsigned char* __restrict__ mask, int j,
                                        float r0, float r1, float r2, float r3) {
    const uchar4 n4 = *reinterpret_cast<const uchar4*>(mask + j);
    if (!(n4.x | n4.y | n4.z | n4.w)) return 0.f;
    const float4 q = __ldg(reinterpret_cast<const float4*>(z + j));
    float rho[KK], w0, w1, w2, w3;
    irs_gmm_eval_t<KK>(gl, q.x, rho, w0);
    irs_gmm_eval_t<KK>(gl, q.y, rho, w1);
    irs_gmm_eval_t<KK>(gl, q.z, rho, w2);
    irs_gmm_eval_t<KK>(gl, q.w, rho, w3);
    return (n4.x ? r0 * (q.x * q.x * w0) : 0.f) + (n4.y ? r1 * (q.y * q.y * w1) : 0.f) + (n4.z ? r2 * (q.z * q.z * w2) : 0.f) +
           (n4.w ? r3 * (q.w * q.w * w3) : 0.f);
}

template <int KK>
__device__ __forceinline__ void gmm_chain_accumulate(const IrsGmm& gl, const float* __restrict__ z,
                                                     const unsigned char* __restrict__ mask, bool vd, IrsDims d, int block,
                                                     int nblocks, float (&acc)[IRS_SUM_COUNT], float4* __restrict__ R) {
    const int V = (int)d.V(), sy = d.W, sz = d.W * d.H;
    auto own = [&](float zi, bool on) {   // all sums of one voxel (branch-free: off-mask results are discarded); returns r
        float rho[KK], wp;
        const float lp = irs_gmm_eval_t<KK>(gl, zi, rho, wp);
        const float z2 = zi * zi, r = on ? z2 * wp : 0.f;
        acc[IRS_SUM_NLL] -= on ? lp : 0.f;
        acc[IRS_SUM_RR] += r * r;
#pragma unroll
        for (int k = 0; k < KK; ++k) if (k < gl.K) {
            acc[IRS_SUM_RHO + k] += on ? rho[k] : 0.f;
            acc[IRS_SUM_Q + k] += on ? rho[k] * z2 * gl.prec[k] : 0.f;
        }
        return r;
    };
    auto res = [&](float zi) {   // residual only (a forward neighbour outside the brick)
        float rho[KK], wp;
        irs_gmm_eval_t<KK>(gl, zi, rho, wp);
        return zi * zi * wp;
    };
    // sum_e r_e * r(neighbour e) with the neighbours at j (brick faces only: kept out of line so that the kernel carries one
    // copy of the four side-by-side evaluations instead of two per path -- the code had outgrown the instruction cache)
    auto halo4 = [&](int j, float r0, float r1, float r2, float r3) { return gmm_halo4<KK>(gl, z, mask, j, r0, r1, r2, r3); };
    const bool vec = d.W >= 4 && (512 % d.W) == 0 && blockDim.x == WALK_T &&
                     ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(mask)) & 15) == 0;
    if (vec) {
        const int w4 = d.W / 4, rows = 512 / d.W;                 // float4 per row, rows of a plane per brick
        const int zz = threadIdx.x >> 7, u = threadIdx.x & 127, row = u / w4, x4 = u - row * w4;
        const int by = (d.H + rows - 1) / rows, bz = (d.D + WALK_PL - 1) / WALK_PL;
        for (int brick = block; brick < by * bz; brick += nblocks) {
            const int y = (brick % by) * rows + row, zc = (brick / by) * WALK_PL + zz;
            const bool valid = y < d.H && zc < d.D;
            const int i = (zc * d.H + y) * d.W + 4 * x4;
            float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) {
                const uchar4 m4 = *reinterpret_cast<const uchar4*>(mask + i);
                if (m4.x | m4.y | m4.z | m4.w) {
                    const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + i));
                    r4.x = own(z4.x, m4.x != 0);
                    r4.y = own(z4.y, m4.y != 0);
                    r4.z = own(z4.z, m4.z != 0);
                    r4.w = own(z4.w, m4.w != 0);
                }
            }
            if (!vd) continue;
            R[threadIdx.x] = r4;
            __syncthreads();
            if (r4.x != 0.f || r4.y != 0.f || r4.z != 0.f || r4.w != 0.f) {   // an exactly zero residual contributes nothing
                const float nx = x4 + 1 < w4 ? R[threadIdx.x + 1].x : 0.f;
                acc[IRS_SUM_RW] += r4.x * r4.y + r4.y * r4.z + r4.z * r4.w + r4.w * nx;
                if (y < d.H - 1) {
                    if (row + 1 < rows) {
                        const float4 q = R[threadIdx.x + w4];
                        acc[IRS_SUM_RH] += r4.x * q.x + r4.y * q.y + r4.z * q.z + r4.w * q.w;
                    } else {
                        acc[IRS_SUM_RH] += halo4(i + sy, r4.x, r4.y, r4.z, r4.w);
                    }
                }
                if (zc < d.D - 1) {
                    if (zz + 1 < WALK_PL) {
                        const float4 q = R[threadIdx.x + 128];
                        acc[IRS_SUM_RD] += r4.x * q.x + r4.y * q.y + r4.z * q.z + r4.w * q.w;
                    } else {
                        acc[IRS_SUM_RD] += halo4(i + sz, r4.x, r4.y, r4.z, r4.w);
                    }
                }
            }
            __syncthreads();   // R is rewritten by the next brick
        }
    } else {
        for (int i = block * blockDim.x + threadIdx.x; i < V; i += nblocks * blockDim.x) {
            if (!mask[i]) continue;
            const float r = own(z[i], true);
            if (!vd) continue;
            const int x = i % d.W, y = (i / d.W) % d.H, zc = i / sz;
            if (x < d.W - 1 && mask[i + 1]) acc[IRS_SUM_RW] += r * res(z[i + 1]);
            if (y < d.H - 1 && mask[i + sy]) acc[IRS_SUM_RH] += r * res(z[i + sy]);
            if (zc < d.D - 1 && mask[i + sz]) acc[IRS_SUM_RD] += r * res(z[i + sz]);
        }
    }
}

template <bool SERIAL, int KK>
__global__ void __launch_bounds__(WALK_T, 1)
gmm_chain_walk_kernel(const float* __restrict__ z_all, const unsigned char* __restrict__ mask, double* __restrict__ hyper_all,
                      long long hyper_stride, IrsHyperCfg cfg, int frozen, double* __restrict__ partials_all,
                      long long partials_stride, unsigned int* __restrict__ counters, unsigned int* __restrict__ ticket,
                      double* __restrict__ stats_all, float* __restrict__ tables_all, int C, IrsDims d) {
    __shared__ IrsGmm g;
    __shared__ double sh[IRS_SUM_COUNT * 32];
    __shared__ double total[IRS_SUM_COUNT];
    __shared__ float4 R[WALK_T];
    __shared__ double alpha_sh;
    const long long V = d.V();
    const int c_first = SERIAL ? 0 : blockIdx.y, c_end = SERIAL ? C : blockIdx.y + 1;
    const int n_used = 5 + IRS_MAX_K + cfg.K;   // the RHO block is padded to IRS_MAX_K slots; Q slots beyond K stay unused
    for (int c = c_first; c < c_end; ++c) {
        double* hyper = hyper_all + (size_t)c * hyper_stride;
        if (SERIAL && c > 0) {
            // chain c - 1 has stepped the shared mixture; its table (written before the ticket was released) is the one
            // this chain evaluates with
            if (threadIdx.x == 0) while (ld_acquire_u32(ticket) < (unsigned int)c) {}
            __syncthreads();
            if (threadIdx.x < 2 * IRS_MAX_K) {
                const float t = __ldcg(tables_all + (size_t)(c - 1) * 16 + threadIdx.x);
                if (threadIdx.x < IRS_MAX_K) g.lw[threadIdx.x] = t; else g.prec[threadIdx.x - IRS_MAX_K] = t;
            }
            if (threadIdx.x == 0) g.K = cfg.K;
        } else if (threadIdx.x == 0) {
            irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, cfg.K, g);
        }
        __syncthreads();
        const IrsGmm gl = g;
        float acc[IRS_SUM_COUNT];
#pragma unroll
        for (int k = 0; k < IRS_SUM_COUNT; ++k) acc[k] = 0.f;
        const float* z = z_all + (size_t)c * V;
        gmm_chain_accumulate<KK>(gl, z, mask, cfg.virtual_decimation != 0, d, blockIdx.x, gridDim.x, acc, R);
        double blk[IRS_SUM_COUNT];
        irs_block_sum<IRS_SUM_COUNT>(acc, blk, sh);
        if (irs_grid_sum<IRS_SUM_COUNT>(blk, partials_all + (size_t)c * partials_stride, counters + c, total, n_used)) {
            // the last CTA to arrive: virtual decimation factor, Adam step (one lane per parameter), the chain's table
            if (threadIdx.x < 32) {
                const int lane = threadIdx.x;
                const double alpha32 = irs_round_f32(cfg.virtual_decimation ? irs_vd_alpha(total, cfg.n_mask) : 1.0);
                gmm_finalize_warp(hyper, cfg, total, alpha32, frozen != 0, tables_all + (size_t)c * 16,
                                  stats_all + (size_t)c * IRS_STAT_SIZE);
                if (SERIAL) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) st_release_u32(ticket, c + 1 < C ? (unsigned int)(c + 1) : 0u);   // the last chain leaves it zero
                }
            }
        }
        __syncthreads();   // `g`, `sh`, `total`, `R` are reused by the next chain
    }
}

// g_z = alpha_c z sum_k rho_k prec_k on the mask (dL/dz of alpha * NLL with the chain's UPDATED mixture), and the
// data term alpha_c * NLL_c for logging
__global__ void __launch_bounds__(256)
gmm_grad_kernel(const float* __restrict__ z_all, const unsigned char* __restrict__ mask,
                const float* __restrict__ tables, int K, double* __restrict__ stats, float* __restrict__ g_all,
                double* __restrict__ partials, unsigned int* __restrict__ counters, IrsDims d) {
    __shared__ double sh[32];
    __shared__ double total[1];
    const int c = blockIdx.y;
    const long long V = d.V();
    IrsGmm g;
    g.K = K;
#pragma unroll
    for (int k = 0; k < IRS_MAX_K; ++k) { g.lw[k] = __ldg(tables + c * 16 + k); g.prec[k] = __ldg(tables + c * 16 + 8 + k); }
    const float alpha = (float)stats[(size_t)c * IRS_STAT_SIZE + IRS_STAT_ALPHA];
    const float* z = z_all + (size_t)c * V;
    float* go = g_all + (size_t)c * V;
    float nll = 0.f;
    auto one = [&](auto kk_tag, float zi, bool on) {   // branch-free like gmm_stats_a_kernel
        constexpr int KK = decltype(kk_tag)::value;
        float rho[KK], wp;
        const float lp = irs_gmm_eval_t<KK>(g, zi, rho, wp);
        nll -= on ? lp : 0.f;
        return on ? alpha * zi * wp : 0.f;
    };
    const bool vec = V % 4 == 0 && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(mask) | reinterpret_cast<uintptr_t>(go)) & 15) == 0;
    auto sweep = [&](auto kk_tag) {
        if (vec) {
            const int Vi = (int)V;
            for (int i = (blockIdx.x * blockDim.x + threadIdx.x) * 4; i < Vi; i += gridDim.x * blockDim.x * 4) {
                const uchar4 m4 = *reinterpret_cast<const uchar4*>(mask + i);
                float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m4.x | m4.y | m4.z | m4.w) {
                    const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + i));
                    g4.x = one(kk_tag, z4.x, m4.x != 0);
                    g4.y = one(kk_tag, z4.y, m4.y != 0);
                    g4.z = one(kk_tag, z4.z, m4.z != 0);
                    g4.w = one(kk_tag, z4.w, m4.w != 0);
                }
                *reinterpret_cast<float4*>(go + i) = g4;
            }
        } else {
            for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x)
                go[i] = mask[i] ? one(kk_tag, z[i], true) : 0.f;
        }
    };
    if (K <= 4) sweep(std::integral_constant<int, 4>{});
    else sweep(std::integral_constant<int, IRS_MAX_K>{});
    double blk[1];
    irs_block_sum<1>(&nll, blk, sh);
    if (irs_grid_sum<1>(blk, partials + (size_t)c * gridDim.x, counters + c, total)) {
        if (threadIdx.x == 0) stats[(size_t)c * IRS_STAT_SIZE + IRS_STAT_DATA] = (double)alpha * total[0];
    }
}

// op-level mixture log-density: logp, d logp / dz and weighted parameter gradients
__global__ void __launch_bounds__(256)
gmm_log_pdf_kernel(const float* __restrict__ z, long long n, IrsGmm g, float* __restrict__ logp, float* __restrict__ dz,
                   const float* __restrict__ weights, double* __restrict__ g_params, double* __restrict__ partials,
                   unsigned int* __restrict__ counter) {
    __shared__ double sh[2 * IRS_MAX_K * 32];
    __shared__ double total[2 * IRS_MAX_K];
    float acc[2 * IRS_MAX_K];
#pragma unroll
    for (int k = 0; k < 2 * IRS_MAX_K; ++k) acc[k] = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float rho[IRS_MAX_K], wp;
        const float zi = z[i];
        const float lp = irs_gmm_eval(g, zi, rho, wp);
        if (logp != nullptr) logp[i] = lp;
        if (dz != nullptr) dz[i] = -zi * wp;
        if (g_params != nullptr) {
            const float w = weights ? weights[i] : 1.f;
#pragma unroll
            for (int k = 0; k < IRS_MAX_K; ++k) if (k < g.K) {
                acc[k] += w * rho[k] * (zi * zi * g.prec[k] - 1.f);  // d logp / d log_std_k
                acc[IRS_MAX_K + k] += w * rho[k];                     // -> d logp / d logits_j = rho_j - pi_j (host adds pi)
            }
        }
    }
    if (g_params == nullptr) return;
    double blk[2 * IRS_MAX_K];
    irs_block_sum<2 * IRS_MAX_K>(acc, blk, sh);
    if (irs_grid_sum<2 * IRS_MAX_K>(blk, partials, counter, total)) {
        if (threadIdx.x < 2 * IRS_MAX_K) g_params[threadIdx.x] = total[threadIdx.x];
    }
}

// virtual decimation factor from an already rescaled residual field r (the second half of the reference's two-call
// sequence rescale_residuals -> calc_VD_factor, utils/util.py:446-485)
__global__ void __launch_bounds__(256)
vd_from_residual_kernel(const float* __restrict__ r, const unsigned char* __restrict__ mask, double* __restrict__ alpha,
                        double* __restrict__ partials, unsigned int* __restrict__ counter, IrsDims d) {
    __shared__ double sh[5 * 32];
    __shared__ double total[5];
    const long long V = d.V(), sy = d.W, sz = (long long)d.W * d.H;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};  // count, sum r^2, sum r r(+D), sum r r(+H), sum r r(+W)
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < V; i += (long long)gridDim.x * blockDim.x) {
        if (!mask[i]) continue;
        const int x = (int)(i % d.W), y = (int)((i / d.W) % d.H), zc = (int)(i / sz);
        const float ri = r[i];
        acc[0] += 1.f;
        acc[1] += ri * ri;
        if (zc < d.D - 1 && mask[i + sz]) acc[2] += ri * r[i + sz];
        if (y < d.H - 1 && mask[i + sy]) acc[3] += ri * r[i + sy];
        if (x < d.W - 1 && mask[i + 1]) acc[4] += ri * r[i + 1];
    }
    double blk[5];
    irs_block_sum<5>(acc, blk, sh);
    if (!irs_grid_sum<5>(blk, partials, counter, total)) return;
    if (threadIdx.x != 0) return;
    double sums[IRS_SUM_COUNT] = {0};
    sums[IRS_SUM_RR] = total[1]; sums[IRS_SUM_RD] = total[2]; sums[IRS_SUM_RH] = total[3]; sums[IRS_SUM_RW] = total[4];
    *alpha = irs_vd_alpha(sums, total[0]);
}

// sum, sum of squares and count over the mask (mixture initialisation: reference trainer/trainer.py:537-541)
__global__ void __launch_bounds__(256)
masked_moments_kernel(const float* __restrict__ z, const unsigned char* __restrict__ mask, long long n,
                      double* __restrict__ out, double* __restrict__ partials, unsigned int* __restrict__ counter) {
    __shared__ double sh[3 * 32];
    __shared__ double total[3];
    // shifted by the first masked value would be better conditioned; residuals are O(1) so plain sums in double suffice
    double s = 0.0, s2 = 0.0, cnt = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (mask[i]) { const double v = (double)z[i]; s += v; s2 += v * v; cnt += 1.0; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s = irs_warp_sum(s); s2 = irs_warp_sum(s2); cnt = irs_warp_sum(cnt);
    if (lane == 0) { sh[warp] = s; sh[32 + warp] = s2; sh[64 + warp] = cnt; }
    __syncthreads();
    double blk[3] = {0.0, 0.0, 0.0};
    if (threadIdx.x == 0) {
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { blk[0] += sh[w]; blk[1] += sh[32 + w]; blk[2] += sh[64 + w]; }
    }
    __syncthreads();
    if (irs_grid_sum<3>(blk, partials, counter, total)) {
        if (threadIdx.x == 0) {
            const double m = total[0] / total[2];
            out[0] = m;
            out[1] = sqrt(fmax(0.0, (total[1] - total[2] * m * m) / (total[2] - 1.0)));
            out[2] = total[2];
        }
    }
}

}  // namespace

int irs_data_blocks(IrsDims d) {
    // 4 CTAs per SM x 148 SMs: enough loads in flight, short final reduction; 2 per SM up to 128^3, where the final
    // reduction over the blocks is a visible part of these latency-bound kernels (measured 48 vs 51 us for the mixture step)
    const int limit = d.V() <= 128ll * 128 * 128 ? 296 : 592;
    long long b = (d.V() + 255) / 256;
    return (int)(b < limit ? b : limit);
}

int irs_launch_lcc_fwd(const float* im, const float* zF, int s, float* a, float* rs, float* z, int C, IrsDims d,
                       cudaStream_t st) {
    IRS_TRY(launch_box<BOX_FWD_MEAN>(im, nullptr, nullptr, 1.f, a, nullptr, s, C, d, st));
    return launch_box<BOX_FWD_VAR>(a, zF, nullptr, 1.f, rs, z, s, C, d, st);
}

int irs_launch_lcc_bwd(const float* g_z, float g_sign, const float* a, const float* rs, int s, float* work, float* g_im,
                       int C, IrsDims d, cudaStream_t st, float* warp_grad) {
    IRS_TRY(launch_box<BOX_BWD_VAR>(g_z, a, rs, g_sign, work, nullptr, s, C, d, st));
    if (warp_grad != nullptr) return launch_box<BOX_BWD_MEAN_WARP>(work, nullptr, nullptr, 1.f, warp_grad, nullptr, s, C, d, st);
    return launch_box<BOX_BWD_MEAN>(work, nullptr, nullptr, 1.f, g_im, nullptr, s, C, d, st);
}

// totals: IRS_SUM_COUNT doubles of scratch; r_scratch: V floats (needed when the VD factor is recomputed)
int irs_launch_gmm_stats_step(const float* z, const unsigned char* mask, double* hyper, const IrsHyperCfg& cfg,
                              double* partials, unsigned int* counter, double* stats_row, float* table_out,
                              const double* alpha_fixed, float* r_scratch, double* totals, IrsDims d, cudaStream_t st) {
    const int V = (int)d.V();
    if (!cfg.virtual_decimation || alpha_fixed != nullptr) {
        gmm_stats_a_kernel<true><<<irs_data_blocks(d), 256, 0, st>>>(z, mask, hyper, cfg, partials, counter, nullptr, nullptr,
                                                                    stats_row, table_out, alpha_fixed, V);
        return (int)cudaGetLastError();
    }
    if (!r_scratch || !totals) return IRS_ERR_BAD_ARG;
    gmm_stats_a_kernel<false><<<irs_data_blocks(d), 256, 0, st>>>(z, mask, hyper, cfg, partials, counter, r_scratch, totals,
                                                                 stats_row, table_out, nullptr, V);
    gmm_stats_b_kernel<<<irs_data_blocks(d), 256, 0, st>>>(r_scratch, hyper, cfg, partials, counter, totals, stats_row,
                                                          table_out, d);
    return (int)cudaGetLastError();
}

// every chain's mixture statistics / virtual decimation factor / Adam step / table in one launch.
// hyper_stride = 0: the shared mixture of the reference, chains in order (persistent grid, tickets); otherwise one parameter
// block per chain (or `frozen`: no Adam step), chains in parallel.  counters: C per-chain counters followed by the ticket.
int irs_launch_gmm_chain_walk(const float* z, const unsigned char* mask, double* hyper, long long hyper_stride,
                              const IrsHyperCfg& cfg, int frozen, double* partials, long long partials_stride,
                              unsigned int* counters, double* stats, float* tables, int C, IrsDims d, cudaStream_t st) {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 148;
    }
    const long long per_pass = (long long)WALK_T * 4;          // voxels one CTA covers per sweep iteration
    long long want = (d.V() + per_pass - 1) / per_pass;
    const bool serial = hyper_stride == 0 && !frozen;
    if (serial) {
        const int G = (int)(want < sms ? want : sms);           // all CTAs resident: they wait for each other
        if ((long long)G * IRS_SUM_COUNT > partials_stride) return IRS_ERR_WORKSPACE;
        // Cooperative launch: the CTAs wait for each other (tickets), so they must all be resident together.  On an otherwise idle
        // GPU a plain launch of <= one CTA per SM would do, but two samplers driving the same GPU from two streams could each get a
        // part of the SMs and wait forever; a cooperative grid is scheduled as a whole or not at all (and is graph-capturable).
        const int frozen0 = 0;
        const long long hs0 = 0;
        unsigned int* ticket = counters + C;
        void* args[] = {(void*)&z, (void*)&mask, (void*)&hyper, (void*)&hs0, (void*)&cfg, (void*)&frozen0, (void*)&partials,
                        (void*)&partials_stride, (void*)&counters, (void*)&ticket, (void*)&stats, (void*)&tables, (void*)&C, (void*)&d};
        const void* fn = cfg.K <= 4 ? (const void*)gmm_chain_walk_kernel<true, 4> : (const void*)gmm_chain_walk_kernel<true, IRS_MAX_K>;
        cudaError_t e = cudaLaunchCooperativeKernel(fn, dim3(G), dim3(WALK_T), args, 0, st);
        if (e != cudaSuccess) return (int)e;
    } else {
        long long per_chain = (2LL * sms + C - 1) / C;          // about two waves of CTAs over all chains
        if (per_chain < 1) per_chain = 1;
        if (want > per_chain) want = per_chain;
        if (want * IRS_SUM_COUNT > partials_stride) return IRS_ERR_WORKSPACE;
        dim3 grid((unsigned)want, C);
        if (cfg.K <= 4)
            gmm_chain_walk_kernel<false, 4><<<grid, WALK_T, 0, st>>>(z, mask, hyper, hyper_stride, cfg, frozen, partials,
                                                                    partials_stride, counters, counters + C, stats, tables, C, d);
        else
            gmm_chain_walk_kernel<false, IRS_MAX_K><<<grid, WALK_T, 0, st>>>(z, mask, hyper, hyper_stride, cfg, frozen, partials,
                                                                            partials_stride, counters, counters + C, stats,
                                                                            tables, C, d);
    }
    return (int)cudaGetLastError();
}

int irs_launch_vd_alpha(const float* z, const unsigned char* mask, double* hyper, const IrsHyperCfg& cfg,
                        double* partials, unsigned int* counter, double* stats_row, IrsDims d, cudaStream_t st) {
    IrsGmm dummy;
    dummy.K = cfg.K;
    gmm_stats_kernel<2><<<irs_data_blocks(d), 256, 0, st>>>(z, mask, hyper, dummy, cfg, partials, counter, stats_row,
                                                           nullptr, nullptr, nullptr, d);
    return (int)cudaGetLastError();
}

// log_std <- linspace(log(sigma/100), log(5 sigma), K), sigma = moments[1]      (reference model/loss.py:61-65)
// ssd: the single Gaussian of the SSD data term starts at the residuals' own scale, log sigma (build-defined; the one-point
// linspace would start at sigma / 100)
__global__ void gmm_init_params_kernel(double* hyper, const double* moments, int K, int ssd) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const double sigma = moments[1];
    const double lo = log(sigma / 100.0), hi = log(sigma * 5.0);
    for (int k = 0; k < K; ++k) {
        // torch.linspace in fp32
        const double t = ssd ? log(sigma) : (K > 1 ? lo + (hi - lo) * (double)k / (double)(K - 1) : lo);
        hyper[IRS_HYPER_LOG_STD + k] = irs_round_f32(t);
    }
}

int irs_launch_gmm_init_params(double* hyper, const double* moments, int K, int ssd, cudaStream_t st) {
    gmm_init_params_kernel<<<1, 32, 0, st>>>(hyper, moments, K, ssd);
    return (int)cudaGetLastError();
}

int irs_launch_gmm_grad(const float* z, const unsigned char* mask, const float* tables, int K, double* stats, float* g,
                        double* partials, unsigned int* counters, int C, IrsDims d, cudaStream_t st) {
    dim3 grid(irs_data_blocks(d), C);
    gmm_grad_kernel<<<grid, 256, 0, st>>>(z, mask, tables, K, stats, g, partials, counters, d);
    return (int)cudaGetLastError();
}

static int table_from_host(const float* gmm_host, int K, IrsGmm& g) {
    if (!gmm_host || K < 1 || K > IRS_MAX_K) return IRS_ERR_BAD_ARG;
    double ls[IRS_MAX_K], lg[IRS_MAX_K];
    for (int k = 0; k < K; ++k) { ls[k] = gmm_host[k]; lg[k] = gmm_host[K + k]; }
    irs_gmm_table(ls, lg, K, g);
    return IRS_OK;
}

extern "C" int irs_lcc_normalise(const float* im, int s, float* a, float* rs, float* zn, int C, int D, int H, int W,
                                 void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!im || !a || s < 1 || s > 3) return IRS_ERR_BAD_ARG;
    return irs_launch_lcc_fwd(im, nullptr, s, a, rs, zn, C, IrsDims{D, H, W}, (cudaStream_t)stream);
}

extern "C" int irs_lcc_normalise_bwd(const float* g_zn, const float* a, const float* rs, int s, float* work,
                                     float* g_im, int C, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(C, D, H, W);
    if (!g_zn || !a || !rs || !work || !g_im || s < 1 || s > 3) return IRS_ERR_BAD_ARG;
    return irs_launch_lcc_bwd(g_zn, 1.f, a, rs, s, work, g_im, C, IrsDims{D, H, W}, (cudaStream_t)stream);
}

extern "C" int irs_gmm_log_pdf(const float* z, long long n, const float* gmm_host, int K, float* logp, float* dz,
                               const float* weights, double* g_params, double* partials, unsigned int* counter,
                               void* stream) {
    if (!z || n < 1) return IRS_ERR_BAD_ARG;
    if (g_params && (!partials || !counter)) return IRS_ERR_BAD_ARG;
    IrsGmm g;
    IRS_TRY(table_from_host(gmm_host, K, g));
    long long b = (n + 255) / 256;
    const int blocks = (int)(b < 1184 ? b : 1184);
    gmm_log_pdf_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(z, n, g, logp, dz, weights, g_params, partials, counter);
    return (int)cudaGetLastError();
}

extern "C" int irs_vd_factor(const float* z, const unsigned char* mask, const float* gmm_host, int K, double* alpha,
                             double* partials, unsigned int* counter, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(1, D, H, W);
    if (!z || !mask || !alpha || !partials || !counter) return IRS_ERR_BAD_ARG;
    IrsGmm g;
    IRS_TRY(table_from_host(gmm_host, K, g));
    IrsHyperCfg cfg = {};
    cfg.K = K;
    cfg.virtual_decimation = 1;
    IrsDims d{D, H, W};
    // n_mask is not known on the host: the kernel recovers it as sum_k sum rho_k (responsibilities sum to 1 per voxel)
    cfg.n_mask = -1.0;
    gmm_stats_kernel<1><<<irs_data_blocks(d), 256, 0, (cudaStream_t)stream>>>(z, mask, nullptr, g, cfg, partials, counter,
                                                                             nullptr, nullptr, alpha, nullptr, d);
    return (int)cudaGetLastError();
}

int irs_launch_masked_moments(const float* z, const unsigned char* mask, long long n, double* out, double* partials,
                              unsigned int* counter, cudaStream_t st) {
    long long b = (n + 255) / 256;
    const int blocks = (int)(b < 1184 ? b : 1184);
    masked_moments_kernel<<<blocks, 256, 0, st>>>(z, mask, n, out, partials, counter);
    return (int)cudaGetLastError();
}

extern "C" int irs_vd_factor_residual(const float* r, const unsigned char* mask, double* alpha, double* partials,
                                      unsigned int* counter, int D, int H, int W, void* stream) {
    IRS_CHECK_DIMS(1, D, H, W);
    if (!r || !mask || !alpha || !partials || !counter) return IRS_ERR_BAD_ARG;
    IrsDims d{D, H, W};
    vd_from_residual_kernel<<<irs_data_blocks(d), 256, 0, (cudaStream_t)stream>>>(r, mask, alpha, partials, counter, d);
    return (int)cudaGetLastError();
}

extern "C" int irs_masked_mean_std(const float* z, const unsigned char* mask, long long n, double* out,
                                   double* partials, unsigned int* counter, void* stream) {
    if (!z || !mask || !out || !partials || !counter || n < 2) return IRS_ERR_BAD_ARG;
    return irs_launch_masked_moments(z, mask, n, out, partials, counter, (cudaStream_t)stream);
}
