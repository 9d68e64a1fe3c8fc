// irs_kernels.cuh -- internal launchers shared between the translation units of libirsgmcmc.so
#pragma once
#include "irs_common.cuh"
#include "../../include/irsgmcmc.h"
#include "irs_hyper.cuh"

#define IRS_CHECK_DIMS(C, D, H, W)                                                       \
    do {                                                                                 \
        if ((C) < 1 || (D) < 2 || (H) < 2 || (W) < 2) return IRS_ERR_BAD_ARG;            \
        if ((long long)(D) * (H) * (W) > 0x7fffffffLL / 4) return IRS_ERR_UNSUPPORTED;   \
        if ((C) > 65535) return IRS_ERR_UNSUPPORTED;                                     \
    } while (0)

// The reference's SVF maps channel i with 2/(shape[2+i]-1) but unnormalises x with W, z with D (utils/util.py:418-429
// vs ATen): consistent only for cubes, which is all its data loader produces (data_loader/datasets.py:76-83).  The
// voxel-unit integrator is therefore defined for cubic volumes only.
#define IRS_CHECK_CUBE(D, H, W)                                      \
    do {                                                             \
        if ((D) != (H) || (H) != (W)) return IRS_ERR_UNSUPPORTED;    \
    } while (0)

#define IRS_LAUNCH_CHECK()                             \
    do {                                               \
        cudaError_t e__ = cudaGetLastError();          \
        if (e__ != cudaSuccess) return (int)e__;       \
    } while (0)

// Launch with programmatic stream serialisation (PDL): the kernel may be scheduled while its predecessor in the stream
// is still draining, so it MUST call irs_pdl_wait() (irs_tma.cuh) before it touches anything a predecessor wrote or reads.
template <typename... KArgs, typename... Args>
inline cudaError_t irs_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                  Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

#define IRS_TRY(expr)                  \
    do {                               \
        int r__ = (expr);              \
        if (r__ != IRS_OK) return r__; \
    } while (0)

// reference utils/util.py:52-53 then :418-429: ((-2 alpha U + alpha) * 2) / (n - 1), fp32, no contraction
__device__ __forceinline__ float irs_jitter_normalised(float u01, float alpha, int n) {
    float noise = __fadd_rn(__fmul_rn(-2.0f * alpha, u01), alpha);
    return __fdiv_rn(__fmul_rn(noise, 2.0f), (float)(n - 1));
}

// log det J from the nine scaled forward differences J[j][comp] = d T_comp / d x_j: the 3x3 determinant written out with
// the same six products in the same order as the reference (utils/util.py:72-91), then logf.  log_det_j_kernel
// (irs_metrics.cu) and the Jacobian posterior (irs_jacobian.cu) both call it, so they compute the same bits.
__device__ __forceinline__ float irs_log_det_3x3(const float (&J)[3][3]) {
    const float det = J[0][0] * J[1][1] * J[2][2] + J[0][1] * J[1][2] * J[2][0] + J[0][2] * J[1][0] * J[2][1] -
                      J[2][0] * J[1][1] * J[0][2] - J[2][1] * J[1][2] * J[0][0] - J[2][2] * J[1][0] * J[0][1];
    return logf(det);
}

// up to 32 segmentation labels of one per-sample evaluation launch (Dice counts, surface distance)
struct LabelList {
    int n;
    int v[32];
};

struct IrsTaps {
    int n;
    float w[IRS_MAX_TAPS + 1];
};

// where a kernel gets its random numbers from: an explicit array (tests, exact parity) or Philox
struct IrsRng {
    const float* explicit_values;  // (C,3,V) or nullptr
    unsigned long long seed;
    const double* iter_ptr;        // device iteration counter (hyper[IRS_HYPER_ITER]) or nullptr
    unsigned long long iter;       // used when iter_ptr == nullptr
    int chain0;
};

// --- irs_sampler.cu: the fused transition with the chain-summed regulariser hyper-gradients scaled (VI: mean of two samples) ---
int irs_sgld_step_scaled(const irs_sgld_config* cfg, const irs_sgld_buffers* b, void* stream, double reg_grad_scale);

// --- irs_warp.cu: voxel-unit warps used by the fused step ------------------------------------------------------------
// grad != nullptr: also writes d out / d position (C,3,V) -- the warp's adjoint becomes a multiplication (irs_launch_lcc_bwd's
// epilogue, or irs_launch_warp_apply_grad)
int irs_launch_warp_vox_fwd(const float* img, const float* u, IrsRng jit, float alpha, int use_jitter, float* out, int C,
                            IrsDims d, cudaStream_t st, float* grad = nullptr);
int irs_launch_warp_apply_grad(const float* g_out, float sign, float* grad, int C, IrsDims d, cudaStream_t st);
int irs_launch_warp_vox_bwd(const float* img, const float* u, IrsRng jit, float alpha, int use_jitter,
                            const float* g_out, float g_sign, float* g_u, int C, IrsDims d, cudaStream_t st);

// --- irs_svf.cu -------------------------------------------------------------------------------------------------------
// energy != nullptr: the first step may also reduce the regulariser energy of v (one double per chain at energy[c *
// energy_stride]; partials: C * irs_svf_fwd_max_blocks(d) doubles; counters: C zeroed uints); *energy_done tells whether it did
int irs_launch_svf_fwd(const float* v, float* hist, float* maxabs, int n_steps, int C, IrsDims d, cudaStream_t st,
                       double* energy, long long energy_stride, double* partials, unsigned int* counters, int* energy_done);
size_t irs_svf_fwd_max_blocks(IrsDims d);
int irs_launch_svf_bwd(const float* v, const float* hist, const float* maxabs, float* g_u, float* g_work, float* g_v,
                       int n_steps, int gather_radius_max, int C, IrsDims d, cudaStream_t st);

// --- irs_smooth.cu ----------------------------------------------------------------------------------------------------
int irs_launch_langevin(const float* v, const float* sigma, long long sigma_cs, float coef, IrsRng rng, float* out,
                        int C, IrsDims d, cudaStream_t st);
int irs_launch_smooth3(const float* in, float* work, float* out, const IrsTaps& taps, int C, IrsDims d,
                       cudaStream_t st);
// out = S * (v + coef sigma eps); work: (C,3,V) scratch
// irs_langevin_fused: whether the state grid d and the tap count let irs_launch_langevin_smooth3 fuse the noise with the x / y
// passes (two launches instead of four); it also needs 16-byte aligned fields and sigma_cs % 4 == 0
bool irs_langevin_fused(IrsDims d, int n_taps);
int irs_launch_langevin_smooth3(const float* v, const float* sigma, long long sigma_cs, float coef, IrsRng rng, float* work,
                                float* out, const IrsTaps& taps, int C, IrsDims d, cudaStream_t st);
int irs_launch_reg_energy(const float* v, double* energy, long long energy_stride, double* partials,
                          unsigned int* counters, int C, IrsDims d, cudaStream_t st);
int irs_reg_energy_blocks(IrsDims d);
// v <- v - tau * sigma^2 * (g_css + coef_c * dE/dcss);  grad_v = sigma^2 * (...)   (coef read from stats rows)
int irs_launch_sgd_update(float* v, const float* sigma, long long sigma_cs, const float* css, const float* g_css,
                          const double* coef, long long coef_stride, float tau, float* grad_v, int C, IrsDims d,
                          cudaStream_t st);

// --- irs_ffd.cu -------------------------------------------------------------------------------------------------------
// kernels: cfg-style tables, 4 s - 1 taps per axis (D, H, W order); work: irs_ffd_work_floats() floats
int irs_launch_ffd(const float* in, float* out, bool adjoint, const float (*kernels)[32], const int* cps, float* work,
                   int C, IrsDims grid, IrsDims d, cudaStream_t st);

// --- irs_data.cu ------------------------------------------------------------------------------------------------------
int irs_launch_lcc_fwd(const float* im, const float* zF, int s, float* a, float* rs, float* z, int C, IrsDims d,
                       cudaStream_t st);
// warp_grad != nullptr: g_im is not written; the last box pass multiplies it into warp_grad (C,3,V) in place = dL/du
int irs_launch_lcc_bwd(const float* g_z, float g_sign, const float* a, const float* rs, int s, float* work, float* g_im,
                       int C, IrsDims d, cudaStream_t st, float* warp_grad = nullptr);
int irs_data_blocks(IrsDims d);
int irs_launch_gmm_stats_step(const float* z, const unsigned char* mask, double* hyper, const IrsHyperCfg& cfg,
                              double* partials, unsigned int* counter, double* stats_row, float* table_out,
                              const double* alpha_fixed, float* r_scratch, double* totals, IrsDims d, cudaStream_t st);
int irs_launch_gmm_chain_walk(const float* z, const unsigned char* mask, double* hyper, long long hyper_stride,
                              const IrsHyperCfg& cfg, int frozen, double* partials, long long partials_stride,
                              unsigned int* counters, double* stats, float* tables, int C, IrsDims d, cudaStream_t st);
int irs_launch_vd_alpha(const float* z, const unsigned char* mask, double* hyper, const IrsHyperCfg& cfg,
                        double* partials, unsigned int* counter, double* stats_row, IrsDims d, cudaStream_t st);
int irs_launch_gmm_init_params(double* hyper, const double* moments, int K, int ssd, cudaStream_t st);
int irs_launch_masked_moments(const float* z, const unsigned char* mask, long long n, double* out, double* partials,
                              unsigned int* counter, cudaStream_t st);
int irs_launch_gmm_grad(const float* z, const unsigned char* mask, const float* tables, int K, double* stats, float* g,
                        double* partials, unsigned int* counters, int C, IrsDims d, cudaStream_t st);
