// TEST INFRASTRUCTURE ONLY -- never linked into libirsgmcmc.so, never imported by the package.
//
// Runs the library's __host__ __device__ per-voxel arithmetic (csrc/irs_common.cuh, irs_bodies.cuh, irs_hyper.cuh) in
// plain loops on the CPU so that the `-m "not gpu"` tests can check it against the oracle without a GPU.  The CUDA
// kernels call exactly these functions once per thread.
#include <algorithm>
#include <cstring>
#include <vector>

#include "../../irsgmcmc_b200/csrc/irs_bodies.cuh"
#include "../../irsgmcmc_b200/csrc/irs_hyper.cuh"

extern "C" {

void emul_svf_fwd(const float* v, float* hist, float* maxabs, int n_steps, int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    const size_t F = (size_t)C * 3 * V;
    const float scale0 = 1.0f / (float)(1 << n_steps);
    for (int k = 0; k < n_steps; ++k) {
        const float* in = k == 0 ? v : hist + (size_t)(k - 1) * F;
        float* out = hist + (size_t)k * F;
        float m = 0.f;
        for (int c = 0; c < C; ++c)
            for (long long i = 0; i < V; ++i)
                m = fmaxf(m, irs_body_svf_fwd(in + (size_t)c * 3 * V, k == 0 ? scale0 : 1.f, out + (size_t)c * 3 * V, V, i, d));
        maxabs[k] = m;
    }
}

// mode 0: gather with the radius from maxabs; mode 1: scatter form for every step
void emul_svf_bwd(const float* v, const float* hist, const float* maxabs, const float* g_u, float* g_v, int n_steps,
                  int mode, int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    const size_t F = (size_t)C * 3 * V;
    const float scale0 = 1.0f / (float)(1 << n_steps);
    std::vector<float> a(g_u, g_u + F), b(F);
    for (int k = n_steps - 1; k >= 0; --k) {
        const float* in = k == 0 ? v : hist + (size_t)(k - 1) * F;
        const float sc = k == 0 ? scale0 : 1.f;
        const int R = (int)floorf(maxabs[k]) + 1;
        for (int c = 0; c < C; ++c) {
            const size_t off = (size_t)c * 3 * V;
            for (long long i = 0; i < V; ++i)
                irs_body_svf_bwd(in + off, sc, a.data() + off, b.data() + off, mode == 0 ? R : -1, sc, V, i, d);
            if (mode == 1) {
                float* g = b.data() + off;
                for (long long i = 0; i < V; ++i)
                    irs_body_svf_bwd_scatter(in + off, sc, a.data() + off, sc, V, i, d,
                                             [&](long long t, int ch, float val) { g[(size_t)ch * V + t] += val; });
            }
        }
        a.swap(b);
    }
    std::memcpy(g_v, a.data(), sizeof(float) * F);
}

void emul_warp_fwd(const float* im, const float* T, float* out, int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    for (int c = 0; c < C; ++c)
        for (long long i = 0; i < V; ++i) {
            float px, py, pz;
            irs_position_from_T(T + (size_t)c * 3 * V, V, i, d, px, py, pz);
            out[(size_t)c * V + i] = irs_body_warp_fwd(im, px, py, pz, d);
        }
}

void emul_warp_bwd_grid(const float* im, const float* T, const float* g_out, float* g_T, int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    for (int c = 0; c < C; ++c)
        for (long long i = 0; i < V; ++i) {
            float px, py, pz;
            irs_position_from_T(T + (size_t)c * 3 * V, V, i, d, px, py, pz);
            float* g = g_T + (size_t)c * 3 * V;
            irs_body_warp_grad(im, px, py, pz, d, g_out[(size_t)c * V + i], 0.5f * (W - 1), 0.5f * (H - 1), 0.5f * (D - 1),
                               g[i], g[V + i], g[2 * V + i]);
        }
}

void emul_warp_nearest_i16(const short* seg, const float* T, short* out, int C, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    for (int c = 0; c < C; ++c)
        for (long long i = 0; i < V; ++i) out[(size_t)c * V + i] = seg[irs_body_nearest_index(T + (size_t)c * 3 * V, V, i, d)];
}

// energy and its gradient for one (C=1) field (3,D,H,W)
double emul_reg_energy(const float* v, float* grad, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V(), sy = W, sz = (long long)W * H;
    double e = 0.0;
    for (int ch = 0; ch < 3; ++ch) {
        const float* f = v + (size_t)ch * V;
        for (long long i = 0; i < V; ++i) {
            int x, y, z;
            irs_voxel_xyz(i, d, x, y, z);
            const float vj = f[i];
            e += irs_diff_energy(vj, x < W - 1 ? f[i + 1] : 0.f, x, W) + irs_diff_energy(vj, y < H - 1 ? f[i + sy] : 0.f, y, H) +
                 irs_diff_energy(vj, z < D - 1 ? f[i + sz] : 0.f, z, D);
            if (grad)
                grad[(size_t)ch * V + i] =
                    irs_diff_energy_grad(x > 0 ? f[i - 1] : 0.f, vj, x < W - 1 ? f[i + 1] : 0.f, x, W) +
                    irs_diff_energy_grad(y > 0 ? f[i - sy] : 0.f, vj, y < H - 1 ? f[i + sy] : 0.f, y, H) +
                    irs_diff_energy_grad(z > 0 ? f[i - sz] : 0.f, vj, z < D - 1 ? f[i + sz] : 0.f, z, D);
        }
    }
    return e;
}

// statistics pass of one chain with the parameters in `hyper`, then VD factor + Adam step (what gmm_stats_kernel does)
// cfg_d: lr_log_std, lr_logits, lr_decay, beta1, beta2, eps, prior_loc, prior_scale, dirichlet_alpha, n_mask
double emul_gmm_stats_step(const float* z, const unsigned char* mask, double* hyper, int K, int vd, const double* cfg_d,
                           float* table_out, double* sums_out, float* dz_out, int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V(), sy = W, sz = (long long)W * H;
    IrsHyperCfg cfg = {};
    cfg.K = K; cfg.virtual_decimation = vd;
    cfg.lr_log_std = cfg_d[0]; cfg.lr_logits = cfg_d[1]; cfg.lr_decay = cfg_d[2]; cfg.beta1 = cfg_d[3]; cfg.beta2 = cfg_d[4];
    cfg.eps = cfg_d[5]; cfg.gmm_prior_loc = cfg_d[6]; cfg.gmm_prior_scale = cfg_d[7]; cfg.dirichlet_alpha = cfg_d[8];
    cfg.n_mask = cfg_d[9];
    IrsGmm g;
    irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, K, g);
    double sums[IRS_SUM_COUNT] = {0};
    auto r_at = [&](long long i) { return mask[i] ? irs_gmm_vd_residual(g, z[i]) : 0.f; };
    for (long long i = 0; i < V; ++i) {
        if (!mask[i]) continue;
        int x, y, zc;
        irs_voxel_xyz(i, d, x, y, zc);
        float rho[IRS_MAX_K], wp;
        const float lp = irs_gmm_eval(g, z[i], rho, wp);
        const float z2 = z[i] * z[i], r = z2 * wp;
        sums[IRS_SUM_NLL] -= lp;
        sums[IRS_SUM_RR] += r * r;
        if (zc < D - 1) sums[IRS_SUM_RD] += r * r_at(i + sz);
        if (y < H - 1) sums[IRS_SUM_RH] += r * r_at(i + sy);
        if (x < W - 1) sums[IRS_SUM_RW] += r * r_at(i + 1);
        for (int k = 0; k < K; ++k) { sums[IRS_SUM_RHO + k] += rho[k]; sums[IRS_SUM_Q + k] += rho[k] * z2 * g.prec[k]; }
    }
    const double alpha = vd ? irs_round_f32(irs_vd_alpha(sums, cfg.n_mask)) : 1.0;
    irs_gmm_adam_step(hyper, cfg, sums, alpha);
    IrsGmm up;
    irs_gmm_table(hyper + IRS_HYPER_LOG_STD, hyper + IRS_HYPER_LOGITS, K, up);
    for (int k = 0; k < IRS_MAX_K; ++k) { table_out[k] = up.lw[k]; table_out[IRS_MAX_K + k] = up.prec[k]; }
    if (sums_out) std::memcpy(sums_out, sums, sizeof(sums));
    if (dz_out) {  // alpha * dNLL/dz with the UPDATED mixture
        for (long long i = 0; i < V; ++i) {
            float rho[IRS_MAX_K], wp = 0.f;
            if (mask[i]) irs_gmm_eval(up, z[i], rho, wp);
            dz_out[i] = mask[i] ? (float)alpha * z[i] * wp : 0.f;
        }
    }
    return alpha;
}

// virtual decimation factor from the five lag sums (RR, RD, RH, RW at IRS_SUM_RR..): what the device evaluates
double emul_vd_alpha(const double* sums, double n_mask) { return irs_vd_alpha(sums, n_mask); }

// cfg_d: reg_type, learnable, lr0, lr1, lr_decay, beta1, beta2, eps, prior_loc, prior_scale, w_reg, dof, shape, rate
void emul_reg_hyper_step(double* hyper, const double* cfg_d, int C, double* stats) {
    IrsHyperCfg cfg = {};
    cfg.reg_type = (int)cfg_d[0]; cfg.reg_learnable = (int)cfg_d[1]; cfg.lr_reg0 = cfg_d[2]; cfg.lr_reg1 = cfg_d[3];
    cfg.lr_decay = cfg_d[4]; cfg.beta1 = cfg_d[5]; cfg.beta2 = cfg_d[6]; cfg.eps = cfg_d[7]; cfg.reg_prior_loc = cfg_d[8];
    cfg.reg_prior_scale = cfg_d[9]; cfg.w_reg = cfg_d[10]; cfg.dof = cfg_d[11]; cfg.w_reg_prior_shape = cfg_d[12];
    cfg.w_reg_prior_rate = cfg_d[13];
    irs_reg_hyper_step(hyper, cfg, C, stats);
}

// the warp of the fused step (csrc/irs_warp.cu warp_vox_fwd_kernel<true>): position_from_u's arithmetic with explicit
// jitter r (C,3,V; nullptr: none), then irs_inside, the clamp, irs_cell and irs_interp_grad
void emul_warp_vox(const float* img, const float* u, const float* r, float alpha, float* out, float* grad, int C, int D,
                   int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V();
    for (int c = 0; c < C; ++c)
        for (long long i = 0; i < V; ++i) {
            int x, y, z;
            irs_voxel_xyz(i, d, x, y, z);
            const float* uc = u + (size_t)c * 3 * V;
            float px = (float)x + uc[i], py = (float)y + uc[V + i], pz = (float)z + uc[2 * V + i];
            if (r != nullptr) {
                const float* rc = r + (size_t)c * 3 * V;
                px += alpha - 2.0f * alpha * rc[i];
                py += alpha - 2.0f * alpha * rc[V + i];
                pz += alpha - 2.0f * alpha * rc[2 * V + i];
            }
            const float mx = irs_inside(px, W), my = irs_inside(py, H), mz = irs_inside(pz, D);
            const IrsCell cell = irs_cell(irs_clampf(px, 0.f, (float)(W - 1)), irs_clampf(py, 0.f, (float)(H - 1)),
                                          irs_clampf(pz, 0.f, (float)(D - 1)), d);
            float dx, dy, dz;
            out[(size_t)c * V + i] = irs_interp_grad(cell, [&](int k) { return img[k]; }, dx, dy, dz);
            float* g = grad + (size_t)c * 3 * V;
            g[i] = dx * mx; g[V + i] = dy * my; g[2 * V + i] = dz * mz;
        }
}

// one voxel of gmm_grad_kernel: irs_gmm_eval_t<kk> (kk = 4 or IRS_MAX_K) with a table of lw[8], prec[8]; g = alpha z wprec
// and log p on the mask, 0 off it
void emul_gmm_grad(const float* z, const unsigned char* mask, const float* table, int K, int kk, float alpha, float* g,
                   float* lp, long long n) {
    IrsGmm gm;
    gm.K = K;
    for (int k = 0; k < IRS_MAX_K; ++k) { gm.lw[k] = table[k]; gm.prec[k] = table[IRS_MAX_K + k]; }
    for (long long i = 0; i < n; ++i) {
        float rho[IRS_MAX_K], wp;
        const float l = kk == 4 ? irs_gmm_eval_t<4>(gm, z[i], rho, wp) : irs_gmm_eval_t<IRS_MAX_K>(gm, z[i], rho, wp);
        g[i] = mask[i] ? alpha * z[i] * wp : 0.f;
        lp[i] = mask[i] ? l : 0.f;
    }
}

// sgd_update_kernel for one chain (3,D,H,W): grad_v = sigma^2 (g_css + k dE/dcss), v -= tau grad_v (sigma nullptr: 1)
void emul_sgd_update(float* v, const float* sigma, const float* css, const float* g_css, float k, float tau, float* grad_v,
                     int D, int H, int W) {
    IrsDims d{D, H, W};
    const long long V = d.V(), sy = W, sz = (long long)W * H;
    for (int ch = 0; ch < 3; ++ch)
        for (long long i = 0; i < V; ++i) {
            int x, y, z;
            irs_voxel_xyz(i, d, x, y, z);
            const size_t o = (size_t)ch * V + i;
            const float* f = css + (size_t)ch * V;
            const float ge = irs_diff_energy_grad(x > 0 ? f[i - 1] : 0.f, f[i], x < W - 1 ? f[i + 1] : 0.f, x, W)
                           + irs_diff_energy_grad(y > 0 ? f[i - sy] : 0.f, f[i], y < H - 1 ? f[i + sy] : 0.f, y, H)
                           + irs_diff_energy_grad(z > 0 ? f[i - sz] : 0.f, f[i], z < D - 1 ? f[i + sz] : 0.f, z, D);
            const float sg = sigma ? sigma[o] : 1.f;
            const float g = sg * sg * (g_css[o] + k * ge);
            grad_v[o] = g;
            v[o] -= tau * g;
        }
}

void emul_normal3(unsigned long long seed, int n, int chain, unsigned long long iter, float* out) {
    for (int i = 0; i < n; ++i) irs_normal3(seed, (uint32_t)i, (uint32_t)chain, iter, out + 3 * (size_t)i);
}

void emul_uniform3(unsigned long long seed, int n, int chain, unsigned long long iter, float* out) {
    for (int i = 0; i < n; ++i) irs_uniform3(seed, (uint32_t)i, (uint32_t)chain, iter, out + 3 * (size_t)i);
}

void emul_philox(unsigned int c0, unsigned int c1, unsigned int c2, unsigned int c3, unsigned int k0, unsigned int k1,
                 unsigned int* out) {
    IrsU4 r = irs_philox(c0, c1, c2, c3, k0, k1);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

}  // extern "C"

// cubic B-spline FFD (csrc/irs_ffd_body.cuh): the three axis passes of irs_ffd_fwd / irs_ffd_bwd in the same order
#include "../../irsgmcmc_b200/csrc/irs_ffd_body.cuh"

static IrsFfdAxis emul_axis(const float* kernel, int s, int off) {
    IrsFfdAxis ax;
    ax.s = s;
    ax.off = off;
    for (int j = 0; j <= IRS_FFD_MAX_KERNEL; ++j) ax.k[j] = j < 4 * s - 1 ? kernel[j] : 0.f;
    return ax;
}

extern "C" void emul_bspline_axis(const float* in, float* out, int adjoint, long long outer, int g, int n,
                                  long long inner, const float* kernel, int s, int off) {
    const IrsFfdAxis ax = emul_axis(kernel, s, off);
    const long long total = outer * (adjoint ? g : n) * inner;
    if (inner == 1 && !adjoint) {   // ffd_fwd_rows_kernel: one table entry per x, rows marched
        for (int x = 0; x < n; ++x) {
            const IrsFfdEntry e = irs_ffd_entry(x, g, ax);
            for (long long row = 0; row < outer; ++row)
                out[row * n + x] = irs_body_ffd_axis_fwd_tab(in + row * g, 1u, e);
        }
        return;
    }
    if (inner == 1 && adjoint) {    // ffd_bwd_rows_kernel: rb rows staged with the bank-conflict skew, then gathered
        const IrsFfdSkew sk = irs_ffd_make_skew(ax.s);
        const int pitch = irs_ffd_row_pitch(n, sk);
        long long rb = 2048 / n;
        rb = rb < 1 ? 1 : (rb > 16 ? 16 : rb);
        std::vector<float> s_rows((size_t)rb * pitch);
        for (long long r0 = 0; r0 < outer; r0 += rb) {
            const long long here = outer - r0 < rb ? outer - r0 : rb;
            std::fill(s_rows.begin(), s_rows.end(), -1.0e30f);   // a read of an unstaged word would show
            for (long long r = 0; r < here; ++r)
                for (int x = 0; x < n; ++x) s_rows[r * pitch + irs_ffd_skew(x, sk)] = in[(r0 + r) * n + x];
            for (long long e = 0; e < here * g; ++e)
                out[r0 * g + e] = irs_body_ffd_axis_bwd_row(s_rows.data() + (e / g) * pitch, sk, (int)(e % g), n, ax);
        }
        return;
    }
    // like the launcher: groups of four consecutive elements when the total allows it, single elements otherwise
    if (total % 4 == 0) {
        for (unsigned i = 0; i < (unsigned)(total / 4); ++i) {
            if (adjoint) irs_body_ffd_axis_group<4, true>(in, i, g, n, (unsigned)inner, ax, out + 4 * (size_t)i);
            else irs_body_ffd_axis_group<4, false>(in, i, g, n, (unsigned)inner, ax, out + 4 * (size_t)i);
        }
    } else {
        for (unsigned i = 0; i < (unsigned)total; ++i) {
            if (adjoint) irs_body_ffd_axis_group<1, true>(in, i, g, n, (unsigned)inner, ax, out + i);
            else irs_body_ffd_axis_group<1, false>(in, i, g, n, (unsigned)inner, ax, out + i);
        }
    }
}

extern "C" void emul_ffd(const float* in, float* out, int adjoint, const float* kd, const float* kh, const float* kw,
                         int sD, int sH, int sW, int C, int gD, int gH, int gW, int D, int H, int W) {
    std::vector<float> t1((size_t)C * 3 * D * gH * gW), t2((size_t)C * 3 * D * H * gW);
    if (!adjoint) {
        emul_bspline_axis(in, t1.data(), 0, (long long)C * 3, gD, D, (long long)gH * gW, kd, sD, sD);
        emul_bspline_axis(t1.data(), t2.data(), 0, (long long)C * 3 * D, gH, H, gW, kh, sH, sH);
        emul_bspline_axis(t2.data(), out, 0, (long long)C * 3 * D * H, gW, W, 1, kw, sW, sW);
    } else {
        emul_bspline_axis(in, t2.data(), 1, (long long)C * 3 * D * H, gW, W, 1, kw, sW, sW);
        emul_bspline_axis(t2.data(), t1.data(), 1, (long long)C * 3 * D, gH, H, gW, kh, sH, sH);
        emul_bspline_axis(t1.data(), out, 1, (long long)C * 3, gD, D, (long long)gH * gW, kd, sD, sD);
    }
}
