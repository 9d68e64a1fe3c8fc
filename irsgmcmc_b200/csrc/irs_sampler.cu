// irs_sampler.cu -- the fused SGLD transition (reference trainer/trainer.py:291-356), posterior moments
// (utils/util.py:114-120) and the small ABI helpers.
//
// One call enqueues the whole iteration for all chains of this GPU on one stream; every scalar (virtual decimation
// factors, mixture / regulariser hyper-parameters and their Adam state, the Philox offset) stays in device memory, so
// the sequence has no host synchronisation and can be captured in a CUDA graph and replayed.
#include <cstdint>

#include "irs_kernels.cuh"

namespace {

__global__ void __launch_bounds__(256)
ssd_residual_kernel(const float* __restrict__ fixed, const float* __restrict__ warped, float* __restrict__ z,
                    long long V) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const size_t o = (size_t)blockIdx.y * V + i;
    z[o] = fixed[i] - warped[o];
}

// regulariser loss / coefficient / Adam step for all chains, then advance the Philox offset
// mode: IRS_HYPER_REFERENCE (chain-summed gradients, one step on the shared parameters), IRS_HYPER_PER_CHAIN (every chain
// steps its own block), IRS_HYPER_FROZEN (losses and coefficients only)
__global__ void __launch_bounds__(128) reg_hyper_kernel(double* hyper, IrsHyperCfg cfg, int C, double* stats, int mode) {
    __shared__ double s0[128], s1[128];
    double g0 = 0.0, g1 = 0.0;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {   // chains in parallel: each needs a log / exp in fp64
        double a, b;
        double* h = mode == IRS_HYPER_PER_CHAIN ? hyper + (size_t)c * IRS_HYPER_SIZE : hyper;
        irs_reg_chain_terms(h, cfg, stats + (size_t)c * IRS_STAT_SIZE, a, b);
        if (mode == IRS_HYPER_PER_CHAIN) irs_reg_adam(h, cfg, a, b);
        g0 += a; g1 += b;
    }
    s0[threadIdx.x] = g0; s1[threadIdx.x] = g1;
    __syncthreads();
    if (threadIdx.x != 0) return;
    if (mode == IRS_HYPER_REFERENCE) {
        g0 = 0.0; g1 = 0.0;
        for (int t = 0; t < blockDim.x; ++t) { g0 += s0[t]; g1 += s1[t]; }   // fixed order: deterministic
        irs_reg_adam(hyper, cfg, g0 * cfg.reg_grad_scale, g1 * cfg.reg_grad_scale);
    }
    hyper[IRS_HYPER_ITER] += 1.0;
}

// running mean / M2 over samples (Welford); `count` = number of samples already folded in
__global__ void __launch_bounds__(256)
welford_kernel(const float* __restrict__ sample, int n_new, long long n, double count, float* __restrict__ mean,
               float* __restrict__ m2) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float m = mean[i], s = m2[i];
    float cnt = (float)count;
    for (int j = 0; j < n_new; ++j) {
        const float x = sample[(size_t)j * n + i];
        cnt += 1.f;
        const float dlt = x - m;
        m += dlt / cnt;
        s += dlt * (x - m);
    }
    mean[i] = m;
    m2[i] = s;
}

// the same recurrence on four elements per thread (128-bit accesses, the next sample's load in flight while this one is folded
// in): the update of 64 chains at 128^3 reads 2 GB -- as the scalar kernel it ran at 2 TB/s
__global__ void __launch_bounds__(256)
welford_vec_kernel(const float* __restrict__ sample, int n_new, long long n, double count, float* __restrict__ mean,
                   float* __restrict__ m2) {
    const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    float4 m = *reinterpret_cast<const float4*>(mean + i), s = *reinterpret_cast<const float4*>(m2 + i);
    float cnt = (float)count;
    float4 x = __ldg(reinterpret_cast<const float4*>(sample + i));
    for (int j = 0; j < n_new; ++j) {
        float4 nx = x;
        if (j + 1 < n_new) nx = __ldg(reinterpret_cast<const float4*>(sample + (size_t)(j + 1) * n + i));
        cnt += 1.f;
        float d;
        d = x.x - m.x; m.x += d / cnt; s.x += d * (x.x - m.x);
        d = x.y - m.y; m.y += d / cnt; s.y += d * (x.y - m.y);
        d = x.z - m.z; m.z += d / cnt; s.z += d * (x.z - m.z);
        d = x.w - m.w; m.w += d / cnt; s.w += d * (x.w - m.w);
        x = nx;
    }
    *reinterpret_cast<float4*>(mean + i) = m;
    *reinterpret_cast<float4*>(m2 + i) = s;
}

__global__ void __launch_bounds__(256)
welford_std_kernel(const float* __restrict__ m2, double count, float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = sqrtf(m2[i] / (float)(count - 1.0));
}

IrsHyperCfg hyper_cfg(const irs_sgld_config* c) {
    IrsHyperCfg h;
    h.K = c->K; h.virtual_decimation = c->virtual_decimation; h.reg_type = c->reg_type; h.reg_learnable = c->reg_learnable;
    h.lr_log_std = c->lr_log_std; h.lr_logits = c->lr_logits; h.lr_reg0 = c->lr_reg0; h.lr_reg1 = c->lr_reg1;
    h.lr_decay = c->lr_decay; h.beta1 = c->beta1; h.beta2 = c->beta2; h.eps = c->adam_eps;
    h.gmm_prior_loc = c->gmm_scale_prior_loc; h.gmm_prior_scale = c->gmm_scale_prior_scale;
    h.dirichlet_alpha = c->dirichlet_alpha;
    h.reg_prior_loc = c->reg_scale_prior_loc; h.reg_prior_scale = c->reg_scale_prior_scale;
    h.w_reg = c->w_reg; h.dof = c->dof;
    h.w_reg_prior_shape = c->w_reg_prior_shape; h.w_reg_prior_rate = c->w_reg_prior_rate;
    h.n_mask = c->n_mask;
    h.reg_grad_scale = 1.0;
    return h;
}

int check_config(const irs_sgld_config* c) {
    if (!c) return IRS_ERR_BAD_ARG;
    IRS_CHECK_DIMS(c->C, c->D, c->H, c->W);
    IRS_CHECK_CUBE(c->D, c->H, c->W);
    if (c->K < 1 || c->K > IRS_MAX_K) return IRS_ERR_BAD_ARG;
    if (c->data_term != IRS_DATA_LCC && c->data_term != IRS_DATA_SSD) return IRS_ERR_BAD_ARG;
    if (c->data_term == IRS_DATA_LCC && (c->lcc_s < 1 || c->lcc_s > 3)) return IRS_ERR_BAD_ARG;
    if (c->reg_type != IRS_REG_L2 && c->reg_type != IRS_REG_LOGNORMAL) return IRS_ERR_BAD_ARG;
    if (c->n_taps < 0 || c->n_taps > IRS_MAX_TAPS || (c->n_taps > 0 && c->n_taps % 2 == 0)) return IRS_ERR_BAD_ARG;
    if (c->svf_steps < 1 || c->svf_steps > IRS_MAX_SVF_STEPS) return IRS_ERR_BAD_ARG;
    if (!(c->n_mask >= 2.0) || !(c->tau >= 0.0) || c->gather_radius_max < 0) return IRS_ERR_BAD_ARG;
    if (c->hyper_mode < IRS_HYPER_REFERENCE || c->hyper_mode > IRS_HYPER_FROZEN) return IRS_ERR_BAD_ARG;
    if (c->ffd_cps[0] != 0 || c->ffd_cps[1] != 0 || c->ffd_cps[2] != 0) {
        const int n[3] = {c->D, c->H, c->W};
        for (int a = 0; a < 3; ++a) {
            if (c->ffd_cps[a] < 1 || c->ffd_cps[a] > 8 || c->ffd_grid[a] < 2) return IRS_ERR_BAD_ARG;
            // the crop [cps, cps + n) must lie inside the (g - 1) cps + 1 elements of the transposed convolution
            if ((long long)c->ffd_cps[a] + n[a] > (long long)(c->ffd_grid[a] - 1) * c->ffd_cps[a] + 1) return IRS_ERR_BAD_ARG;
        }
        IRS_CHECK_DIMS(c->C, c->ffd_grid[0], c->ffd_grid[1], c->ffd_grid[2]);
    }
    return IRS_OK;
}

inline bool has_ffd(const irs_sgld_config* c) { return c->ffd_cps[0] > 0; }
// one persistent launch for the mixture step of all chains (irs_launch_gmm_chain_walk) instead of two launches per chain.
// Always for the chain-parallel hyper modes.  In the reference mode (chains in order on the shared mixture) the walk wins where
// a chain is small and the two launches are pure latency (measured, 64 chains: 64^3 1.45 vs 1.77 ms; 128^3 3.13 vs 2.56 ms --
// there one CTA per SM under-fills the machine), hence the volume threshold.
inline bool gmm_walk_enabled(const irs_sgld_config* c) {
    if (c->hyper_mode != IRS_HYPER_REFERENCE) return true;
    return (long long)c->D * c->H * c->W <= 96LL * 96 * 96;
}
// the grid the chain state lives on: the control grid with the FFD, the image grid otherwise
inline IrsDims state_dims(const irs_sgld_config* c) {
    return has_ffd(c) ? IrsDims{c->ffd_grid[0], c->ffd_grid[1], c->ffd_grid[2]} : IrsDims{c->D, c->H, c->W};
}

}  // namespace

extern "C" size_t irs_sgld_partials_doubles(const irs_sgld_config* cfg) {
    if (!cfg) return 0;
    IrsDims d{cfg->D, cfg->H, cfg->W};
    size_t per_chain = (size_t)irs_data_blocks(d) * IRS_SUM_COUNT;
    const size_t fwd = irs_svf_fwd_max_blocks(d);   // the first squaring step reduces the regulariser energy
    if (fwd > per_chain) per_chain = fwd;
    const size_t energy = (size_t)irs_reg_energy_blocks(state_dims(cfg));   // stand-alone energy kernel
    if (energy > per_chain) per_chain = energy;
    return (size_t)cfg->C * per_chain;
}

extern "C" int irs_sgld_launches_per_step(const irs_sgld_config* c) {
    if (check_config(c) != IRS_OK) return -1;
    int n = 1;                                   // langevin (fused with the x / y smoothing when the field can be vectorised;
                                                 // pointer alignment is assumed)
    n += c->n_taps > 0 ? (irs_langevin_fused(state_dims(c), c->n_taps) ? 1 : 3) : 0;   // Sobolev: z pass only / z, y, x
    n += (c->W % 4 == 0 && !has_ffd(c)) ? 0 : 1; // regulariser energy (an epilogue of the first squaring step otherwise)
    n += has_ffd(c) ? 6 : 0;                     // B-spline FFD: three axis passes forward, three for the adjoint
    n += c->svf_steps;                           // scaling and squaring
    n += c->svf_steps > 1 ? 1 : 0;               // cell maps of the last four steps, one launch (exits at once below one voxel)
    n += 1;                                      // warp
    n += c->data_term == IRS_DATA_LCC ? 2 : 1;   // LCC boxes / SSD residual
    n += gmm_walk_enabled(c) ? 1 : c->C * (c->virtual_decimation ? 2 : 1);   // mixture statistics + VD factor + Adam of all chains
    n += 1;                                      // dL/dz
    n += c->data_term == IRS_DATA_LCC ? 2 : 0;   // LCC adjoint boxes
    n += c->data_term == IRS_DATA_LCC ? 0 : 1;   // warp adjoint: an epilogue of the last LCC adjoint box pass; SSD: warp_apply_grad
    n += 1;                                      // regulariser hyper step
    n += c->svf_steps + (c->svf_steps < 4 ? c->svf_steps : 4);   // SVF adjoint (gather; the last four steps carry the
                                                                 // early-exit large-displacement scatter companion)
    n += 1;                                      // regulariser gradient + SGD update
    return n;
}

namespace {
struct StageTimer {
    cudaEvent_t ev[IRS_N_STAGES + 1];
    int n;
};
inline void mark(StageTimer* t, cudaStream_t st) {
    if (t != nullptr && t->n <= IRS_N_STAGES) cudaEventRecord(t->ev[t->n++], st);
}
}  // namespace

static int sgld_step_impl(const irs_sgld_config* cfg, const irs_sgld_buffers* b, void* stream, StageTimer* tm,
                          double reg_grad_scale = 1.0) {
    IRS_TRY(check_config(cfg));
    if (!b || !b->v || !b->fixed || !b->moving || !b->mask || !b->css || !b->hist || !b->im_warped || !b->z ||
        !b->scratch1 || !b->field_a || !b->field_b || !b->grad_v || !b->maxabs || !b->hyper || !b->stats ||
        !b->gmm_table || !b->partials || !b->counters)
        return IRS_ERR_BAD_ARG;
    if (cfg->data_term == IRS_DATA_LCC && (!b->lcc_a || !b->lcc_rs)) return IRS_ERR_BAD_ARG;
    if (!b->scratch2) return IRS_ERR_BAD_ARG;
    const bool ffd = has_ffd(cfg);
    if (ffd && (!b->ffd_dense || !b->ffd_grad || !b->ffd_scratch || !b->ffd_work)) return IRS_ERR_BAD_ARG;

    cudaStream_t st = (cudaStream_t)stream;
    const int C = cfg->C;
    const IrsDims d{cfg->D, cfg->H, cfg->W};
    const IrsDims ds = state_dims(cfg);          // v, sigma, eps, css, grad_v live on this grid
    float* smooth_work = ffd ? b->ffd_scratch : b->field_a;
    const float* velocity = ffd ? b->ffd_dense : b->css;   // what scaling and squaring integrates
    const long long V = d.V();
    const size_t F = (size_t)C * 3 * V;
    IrsHyperCfg hc = hyper_cfg(cfg);
    hc.reg_grad_scale = reg_grad_scale;
    const double* iter_ptr = b->hyper + IRS_HYPER_ITER;

    mark(tm, st);
    // (1) Langevin proposal + Sobolev smoothing                                   trainer.py:292-293
    IrsRng rng_l{b->eps, cfg->seed, iter_ptr, 0ull, cfg->chain_offset};
    const float coef = (float)sqrt(2.0 * cfg->tau);
    if (cfg->n_taps > 0) {
        IrsTaps taps;
        taps.n = cfg->n_taps;
        for (int t = 0; t < cfg->n_taps; ++t) taps.w[t] = cfg->taps[t];
        IRS_TRY(irs_launch_langevin_smooth3(b->v, b->sigma, b->sigma_chain_stride, coef, rng_l, smooth_work, b->css, taps, C, ds, st));
    } else {
        IRS_TRY(irs_launch_langevin(b->v, b->sigma, b->sigma_chain_stride, coef, rng_l, b->css, C, ds, st));
    }
    // (1b) control points -> dense velocity field                                  utils/transformation.py:155-164
    if (ffd) IRS_TRY(irs_launch_ffd(b->css, b->ffd_dense, false, cfg->ffd_kernel, cfg->ffd_cps, b->ffd_work, C, ds, d, st));

    mark(tm, st);
    // (2) + (3) scaling and squaring; its first step also reduces the regulariser energy y_c of css from the planes it
    // holds in shared memory (trainer.py:294, 311).  When that kernel cannot run (row pitch not addressable by the TMA
    // unit) the stand-alone energy kernel follows.
    int energy_done = 0;
    // With the FFD the regulariser acts on the control-point field css, not on the field being integrated.
    IRS_TRY(irs_launch_svf_fwd(velocity, b->hist, b->maxabs, cfg->svf_steps, C, d, st,
                               ffd ? nullptr : b->stats + IRS_STAT_ENERGY, IRS_STAT_SIZE, b->partials, b->counters,
                               &energy_done));
    const float* disp = b->hist + (size_t)(cfg->svf_steps - 1) * F;
    mark(tm, st);
    if (!energy_done)
        IRS_TRY(irs_launch_reg_energy(b->css, b->stats + IRS_STAT_ENERGY, IRS_STAT_SIZE, b->partials, b->counters, C, ds, st));

    mark(tm, st);
    // (4) warp the moving image at T (+ jitter)                                   trainer.py:296-300
    IrsRng rng_j{b->jitter_unit, cfg->seed, iter_ptr, 0ull, cfg->chain_offset};
    const float alpha = (float)cfg->jitter_alpha;
    // ... and leave the warp's spatial gradient in field_a (free between the smoothing and the adjoint): stage 8 multiplies
    IRS_TRY(irs_launch_warp_vox_fwd(b->moving, disp, rng_j, alpha, cfg->use_jitter, b->im_warped, C, d, st, b->field_a));

    mark(tm, st);
    // (5) residual map                                                            trainer.py:307
    if (cfg->data_term == IRS_DATA_LCC) {
        IRS_TRY(irs_launch_lcc_fwd(b->im_warped, b->fixed, cfg->lcc_s, b->lcc_a, b->lcc_rs, b->z, C, d, st));
    } else {
        dim3 grid((unsigned)((V + 255) / 256), C);
        ssd_residual_kernel<<<grid, 256, 0, st>>>(b->fixed, b->im_warped, b->z, V);
        IRS_LAUNCH_CHECK();
    }

    mark(tm, st);
    // (6) per chain, in order: VD factor, Adam step on the shared mixture          trainer.py:316-318
    const size_t per_chain = (size_t)irs_data_blocks(d) * IRS_SUM_COUNT;
    if (gmm_walk_enabled(cfg)) {
        IRS_TRY(irs_launch_gmm_chain_walk(b->z, b->mask, b->hyper, cfg->hyper_mode == IRS_HYPER_PER_CHAIN ? IRS_HYPER_SIZE : 0,
                                          hc, cfg->hyper_mode == IRS_HYPER_FROZEN, b->partials, (long long)per_chain,
                                          b->counters, b->stats, b->gmm_table, C, d, st));
    } else {
        for (int c = 0; c < C; ++c) {
            IRS_TRY(irs_launch_gmm_stats_step(b->z + (size_t)c * V, b->mask, b->hyper, hc, b->partials + c * per_chain,
                                              b->counters + c, b->stats + (size_t)c * IRS_STAT_SIZE,
                                              b->gmm_table + (size_t)c * 16, nullptr, b->scratch2 + (size_t)c * V,
                                              b->hyper + IRS_HYPER_SCRATCH, d, st));
        }
    }

    mark(tm, st);
    // (7) dL/dz with each chain's updated mixture + the logged data term          trainer.py:320
    IRS_TRY(irs_launch_gmm_grad(b->z, b->mask, b->gmm_table, cfg->K, b->stats, b->scratch1, b->partials, b->counters, C,
                                d, st));

    mark(tm, st);
    // (8) back through the residual map and the warp -> dL/du_n = dL/dM_w * grad M(p): the product is the epilogue of the
    // last adjoint box pass (utils/registration.py:29-30 backward without a second gather)
    if (cfg->data_term == IRS_DATA_LCC) {
        IRS_TRY(irs_launch_lcc_bwd(b->scratch1, -1.f, b->lcc_a, b->lcc_rs, cfg->lcc_s, b->scratch2, b->scratch1, C, d, st,
                                   b->field_a));
    } else {
        IRS_TRY(irs_launch_warp_apply_grad(b->scratch1, -1.f, b->field_a, C, d, st));
    }

    mark(tm, st);
    // (9) regulariser loss, coefficient and hyper-parameter Adam step              trainer.py:311,334-339,353-354
    reg_hyper_kernel<<<1, 128, 0, st>>>(b->hyper, hc, C, b->stats, cfg->hyper_mode);
    IRS_LAUNCH_CHECK();

    mark(tm, st);
    // (10) SVF adjoint -> dL/dcss (data part)                                      trainer.py:349
    IRS_TRY(irs_launch_svf_bwd(velocity, b->hist, b->maxabs, b->field_a, b->field_b, ffd ? b->ffd_grad : b->grad_v,
                               cfg->svf_steps, cfg->gather_radius_max, C, d, st));
    // (10b) dense gradient -> control points (gathers over each control point's support)
    if (ffd) IRS_TRY(irs_launch_ffd(b->ffd_grad, b->grad_v, true, cfg->ffd_kernel, cfg->ffd_cps, b->ffd_work, C, ds, d, st));

    mark(tm, st);
    // (11) + regulariser gradient, sigma^2 preconditioning, SGD step               utils/functions.py:82-84, trainer.py:351
    IRS_TRY(irs_launch_sgd_update(b->v, b->sigma, b->sigma_chain_stride, b->css, b->grad_v, b->stats + IRS_STAT_REG_COEF,
                                  IRS_STAT_SIZE, (float)cfg->tau, b->grad_v, C, ds, st));
    mark(tm, st);
    return IRS_OK;
}

extern "C" int irs_sgld_step(const irs_sgld_config* cfg, const irs_sgld_buffers* b, void* stream) {
    return sgld_step_impl(cfg, b, stream, nullptr);
}

int irs_sgld_step_scaled(const irs_sgld_config* cfg, const irs_sgld_buffers* b, void* stream, double reg_grad_scale) {
    return sgld_step_impl(cfg, b, stream, nullptr, reg_grad_scale);
}

// Profiling aid (not for graph capture; synchronises): runs one transition eagerly with a CUDA event between the
// stages and writes the IRS_N_STAGES stage durations in milliseconds to ms_host.
extern "C" int irs_sgld_step_profile(const irs_sgld_config* cfg, const irs_sgld_buffers* b, void* stream,
                                     float* ms_host) {
    if (!ms_host) return IRS_ERR_BAD_ARG;
    StageTimer tm;
    tm.n = 0;
    for (int i = 0; i <= IRS_N_STAGES; ++i) {
        cudaError_t e = cudaEventCreate(&tm.ev[i]);
        if (e != cudaSuccess) return (int)e;
    }
    int r = sgld_step_impl(cfg, b, stream, &tm);
    cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
    if (r == IRS_OK && e != cudaSuccess) r = (int)e;
    if (r == IRS_OK) {
        for (int i = 0; i < IRS_N_STAGES; ++i) {
            ms_host[i] = 0.f;
            if (i + 1 < tm.n) cudaEventElapsedTime(&ms_host[i], tm.ev[i], tm.ev[i + 1]);
        }
    }
    for (int i = 0; i <= IRS_N_STAGES; ++i) cudaEventDestroy(tm.ev[i]);
    return r;
}

// Mixture initialisation (reference trainer/trainer.py:529-547): smooth the given velocity sample (no Langevin noise),
// integrate, warp (no jitter), residual map, sigma_hat = std over the mask, log_std = linspace(log sigma_hat/100,
// log 5 sigma_hat, K), VD factor once, then n_warmup Adam steps on the mixture with that factor.
// Uses the chain-0 slices of the step buffers; v_sample is (1,3,D,H,W).
extern "C" int irs_sgld_gmm_init(const irs_sgld_config* cfg, const irs_sgld_buffers* b, const float* v_sample,
                                 int n_warmup, void* stream) {
    IRS_TRY(check_config(cfg));
    if (!b || !v_sample || n_warmup < 0) return IRS_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const IrsDims d{cfg->D, cfg->H, cfg->W};
    const long long V = d.V();
    const IrsHyperCfg hc = hyper_cfg(cfg);
    IrsRng none{nullptr, 0ull, nullptr, 0ull, 0};
    const bool ffd = has_ffd(cfg);
    if (ffd && (!b->ffd_dense || !b->ffd_scratch || !b->ffd_work)) return IRS_ERR_BAD_ARG;
    const IrsDims ds = state_dims(cfg);   // v_sample is (1,3,gD,gH,gW) with the FFD
    float* smooth_work = ffd ? b->ffd_scratch : b->field_a;
    if (cfg->n_taps > 0) {
        IrsTaps taps;
        taps.n = cfg->n_taps;
        for (int t = 0; t < cfg->n_taps; ++t) taps.w[t] = cfg->taps[t];
        IRS_TRY(irs_launch_langevin_smooth3(v_sample, nullptr, 0, 0.f, none, smooth_work, b->css, taps, 1, ds, st));
    } else {
        IRS_TRY(irs_launch_langevin(v_sample, nullptr, 0, 0.f, none, b->css, 1, ds, st));
    }
    if (ffd) IRS_TRY(irs_launch_ffd(b->css, b->ffd_dense, false, cfg->ffd_kernel, cfg->ffd_cps, b->ffd_work, 1, ds, d, st));
    // hist of a single chain is laid out with stride 3V per step when C = 1
    IRS_TRY(irs_launch_svf_fwd(ffd ? b->ffd_dense : b->css, b->hist, b->maxabs, cfg->svf_steps, 1, d, st, nullptr, 0, nullptr,
                               nullptr, nullptr));
    const float* disp = b->hist + (size_t)(cfg->svf_steps - 1) * 3 * V;
    IRS_TRY(irs_launch_warp_vox_fwd(b->moving, disp, none, 0.f, 0, b->im_warped, 1, d, st));
    if (cfg->data_term == IRS_DATA_LCC) {
        IRS_TRY(irs_launch_lcc_fwd(b->im_warped, b->fixed, cfg->lcc_s, b->lcc_a, b->lcc_rs, b->z, 1, d, st));
    } else {
        dim3 grid((unsigned)((V + 255) / 256), 1);
        ssd_residual_kernel<<<grid, 256, 0, st>>>(b->fixed, b->im_warped, b->z, V);
        IRS_LAUNCH_CHECK();
    }
    double* moments = b->stats + IRS_STAT_SIZE - 3;  // last three slots of chain 0's row, overwritten by the next step
    IRS_TRY(irs_launch_masked_moments(b->z, b->mask, V, moments, b->partials, b->counters, st));
    IRS_TRY(irs_launch_gmm_init_params(b->hyper, moments, cfg->K, cfg->data_term == IRS_DATA_SSD, st));
    IRS_TRY(irs_launch_vd_alpha(b->z, b->mask, b->hyper, hc, b->partials, b->counters, b->stats, d, st));
    for (int it = 0; it < n_warmup; ++it)
        IRS_TRY(irs_launch_gmm_stats_step(b->z, b->mask, b->hyper, hc, b->partials, b->counters, b->stats, b->gmm_table,
                                          b->stats + IRS_STAT_ALPHA, nullptr, nullptr, d, st));
    return IRS_OK;
}

extern "C" int irs_welford_update(const float* sample, int n_new, long long n, double count_before, float* mean,
                                  float* m2, void* stream) {
    if (!sample || !mean || !m2 || n_new < 1 || n < 1 || count_before < 0) return IRS_ERR_BAD_ARG;
    const bool vec = (n % 4) == 0 && ((reinterpret_cast<uintptr_t>(sample) | reinterpret_cast<uintptr_t>(mean) |
                                       reinterpret_cast<uintptr_t>(m2)) & 15) == 0;
    if (vec) welford_vec_kernel<<<(unsigned)((n / 4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(sample, n_new, n, count_before, mean, m2);
    else welford_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(sample, n_new, n, count_before, mean, m2);
    return (int)cudaGetLastError();
}

extern "C" int irs_welford_std(const float* m2, double count, float* std_out, long long n, void* stream) {
    if (!m2 || !std_out || n < 1 || count < 2) return IRS_ERR_BAD_ARG;
    welford_std_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(m2, count, std_out, n);
    return (int)cudaGetLastError();
}

extern "C" int irs_abi_version(void) { return IRS_ABI_VERSION; }

extern "C" const char* irs_error_string(int code) {
    switch (code) {
        case IRS_OK: return "ok";
        case IRS_ERR_BAD_ARG: return "irsgmcmc: bad argument (null pointer, size or option out of range)";
        case IRS_ERR_UNSUPPORTED: return "irsgmcmc: unsupported shape or option";
        case IRS_ERR_WORKSPACE: return "irsgmcmc: workspace too small";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "irsgmcmc: unknown error";
    }
}
