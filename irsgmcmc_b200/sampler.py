"""
SGLDSampler -- the fused, graph-captured SGLD registration step for all chains resident on one GPU.

One `step()` == one `Trainer._SGLD_transition` of the reference (trainer/trainer.py:291-356) for `no_chains` chains:
Langevin proposal, Sobolev smoothing, scaling and squaring, jittered warp, LCC/GMM (or SSD) data term with virtual
decimation and the sequential per-chain Adam step on the shared mixture, regulariser with its hyper-parameter Adam
step, backward pass and the preconditioned SGD update -- as one CUDA graph of libirsgmcmc.so kernels with no host
synchronisation.  Kept samples feed on-device Welford moments (replaces the host-side sample buffer +
calc_posterior_statistics, utils/util.py:114-120, trainer/trainer.py:365-366,428-430,458).

PyTorch supplies device memory, streams, CUDA-graph capture and torch.distributed; all arithmetic is in the library.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from .utils.functions import Sobolev_kernel_1D


class SGLDConfig:
    """hyper-parameters of the hot path; defaults are the reference's configs/experiment3/config.json"""

    def __init__(self, data_loss='lcc', no_components=4, s=2, reg_loss='RegLoss_LogNormal', w_reg=1.6,
                 reg_learnable=True, sobolev_enabled=True, sobolev_s=3, sobolev_lambda=0.5, svf_steps=12, tau=0.4,
                 uniform_noise=True, uniform_noise_magnitude=0.1, virtual_decimation=True, lr_log_std=0.2,
                 lr_logits=0.2, lr_reg=0.01, lr_decay=1e-3, betas=(0.9, 0.999), adam_eps=1e-8,
                 gmm_scale_prior=(0.0, 2.3), dirichlet_alpha=0.5, reg_scale_prior=(2.8, 5.0), gather_radius_max=2,
                 seed=123, transformation='SVF_3D', cps=None, hyper_mode='reference'):
        if data_loss not in ('lcc', 'ssd'):
            raise ValueError(f'unknown data loss: {data_loss}')
        if transformation not in ('SVF_3D', 'SVFFD_3D'):
            raise ValueError(f'unknown transformation module: {transformation}')
        if transformation == 'SVFFD_3D':   # configs/experiment5/config_SVFFD_*.json: "cps": [s, s, s]
            if cps is None or len(cps) != 3 or not all(1 <= int(c) <= 8 for c in cps):
                raise ValueError('SVFFD_3D needs cps = three control point spacings between 1 and 8')
            cps = tuple(int(c) for c in cps)
        # 'reference': one mixture / regulariser parameter set shared by all chains, stepped chain after chain (the reference's
        # loop, trainer/trainer.py:316-327,353-354); 'per_chain': every chain owns its parameters (= an independent reference run
        # with one chain each); 'frozen': shared parameters, no Adam steps.  The last two have no dependency between chains.
        if hyper_mode not in _lib.HYPER_MODES:
            raise ValueError(f'unknown hyper_mode: {hyper_mode} (one of {sorted(_lib.HYPER_MODES)})')
        if reg_loss not in ('RegLoss_LogNormal', 'RegLoss_L2'):
            raise ValueError(f'unknown regularisation loss: {reg_loss}')
        self.__dict__.update(locals())
        del self.__dict__['self']
        if data_loss == 'ssd':
            self.no_components = 1


def lognormal_init(w_reg, dof):
    """(loc, log_scale) of RegLoss_LogNormal (reference model/loss.py:300-305, model/distributions.py:171-172)"""
    # nu and w_reg are fp32 tensors in the reference (model/distributions.py:234-236): the rate and its log are fp32
    log_rate = float(torch.log(0.5 * torch.tensor(1.0) * torch.tensor(w_reg, dtype=torch.float32)))
    loc = float(torch.digamma(torch.tensor(0.5 * dof, dtype=torch.float64))) - log_rate
    return loc, math.log(4.0) + math.log(loc)


class SGLDSampler:
    def __init__(self, fixed, moving, no_chains, config=None, device='cuda:0', chain_offset=0, keep_grad=True):
        """
        fixed / moving: the reference's data dicts {'im': f32 (1,1,D,H,W), 'mask': bool (1,1,D,H,W), 'seg': int16}
        (data_loader/datasets.py:117,128,135); only fixed['mask'] gates the data term (trainer/trainer.py:308)
        """
        self.cfg = cfg = config or SGLDConfig()
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('SGLDSampler needs a CUDA device: irsgmcmc_b200 has no CPU path')
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        dev = self.device

        im_f = fixed['im'].to(dev, torch.float32).contiguous()
        im_m = moving['im'].to(dev, torch.float32).contiguous()
        if im_f.dim() != 5 or im_f.shape[:2] != (1, 1) or im_m.shape != im_f.shape:
            raise ValueError('images must have shape (1,1,D,H,W)')
        self.dims = D, H, W = tuple(im_f.shape[2:])
        self.V = V = D * H * W
        self.C = C = int(no_chains)
        self.chain_offset = int(chain_offset)
        self.mask = fixed['mask'].to(dev).contiguous().view(torch.uint8) if fixed['mask'].dtype == torch.bool \
            else fixed['mask'].to(dev, torch.uint8).contiguous()
        self.n_mask = float(self.mask.sum().item())
        self.moving_im = im_m
        self.fixed_im = im_f
        self.moving_seg = moving['seg'].to(dev).contiguous() if 'seg' in moving else None

        f32 = dict(device=dev, dtype=torch.float32)
        if cfg.data_loss == 'lcc':
            # the fixed-image side of the LCC map is constant: computed once (the reference redoes it every iteration)
            a = torch.empty(1, 1, D, H, W, **f32)
            self.fixed_term = torch.empty(1, 1, D, H, W, **f32)
            _lib.check(self.lib.irs_lcc_normalise(_lib.ptr(im_f), cfg.s, _lib.ptr(a), None, _lib.ptr(self.fixed_term),
                                                  1, D, H, W, _lib.stream()))
        else:
            self.fixed_term = im_f

        # with SVFFD_3D the chain state lives on the control grid (data_loader/datasets.py:23-27), everything behind the
        # B-spline FFD on the image grid
        self.ffd = cfg.transformation == 'SVFFD_3D'
        if self.ffd:
            from .utils.transformation import B_spline_1D_kernel
            from .utils.util import get_control_grid_size
            self.state_dims = get_control_grid_size(self.dims, cfg.cps)
            self._ffd_taps = [[float(k) for k in B_spline_1D_kernel(c)] for c in cfg.cps]
        else:
            self.state_dims = self.dims
        gD, gH, gW = self.state_dims

        # state + workspace, allocated once (180 GB HBM: the SVF history is kept rather than recomputed)
        self.v = torch.zeros(C, 3, gD, gH, gW, **f32)
        self.sigma = None
        self.css = torch.empty(C, 3, gD, gH, gW, **f32)
        self.hist = torch.empty(cfg.svf_steps, C, 3, D, H, W, **f32)
        self.im_warped = torch.empty(C, 1, D, H, W, **f32)
        self.z = torch.empty(C, 1, D, H, W, **f32)
        self._lcc_a = torch.empty(C, 1, D, H, W, **f32)
        self._lcc_rs = torch.empty(C, 1, D, H, W, **f32)
        self._scratch1 = torch.empty(C, 1, D, H, W, **f32)
        self._scratch2 = torch.empty(C, 1, D, H, W, **f32)
        self._field_a = torch.empty(C, 3, D, H, W, **f32)
        self._field_b = torch.empty(C, 3, D, H, W, **f32)
        self.grad_v = torch.zeros(C, 3, gD, gH, gW, **f32)
        if self.ffd:
            self._ffd_dense = torch.empty(C, 3, D, H, W, **f32)
            self._ffd_grad = torch.empty(C, 3, D, H, W, **f32)
            self._ffd_scratch = torch.empty(C, 3, gD, gH, gW, **f32)
            self._ffd_work = torch.empty(int(self.lib.irs_ffd_work_floats(C, gD, gH, gW, D, H, W)), **f32)
        self._maxabs = torch.zeros(int(self.lib.irs_svf_maxabs_floats(C, D, H, W, cfg.svf_steps)), **f32)
        self.per_chain = cfg.hyper_mode == 'per_chain'
        # (HYPER_SIZE,) shared block; (C, HYPER_SIZE) with hyper_mode='per_chain' (block 0 carries the iteration counter)
        self.hyper = torch.zeros((C, _lib.HYPER_SIZE) if self.per_chain else (_lib.HYPER_SIZE,), device=dev, dtype=torch.float64)
        self.stats = torch.zeros(C, _lib.STAT_SIZE, device=dev, dtype=torch.float64)
        self._gmm_table = torch.zeros(C, 16, **f32)
        self._counters = torch.zeros(C + 8, device=dev, dtype=torch.int32)
        self.eps_inject = None
        self.jitter_inject = None

        self.dof = 3.0 * V
        if cfg.reg_loss == 'RegLoss_LogNormal':
            loc, log_scale = lognormal_init(cfg.w_reg, self.dof)
            self.hyper[..., _lib.HYPER_REG_P] = loc
            self.hyper[..., _lib.HYPER_REG_P + 1] = log_scale
        else:
            self.hyper[..., _lib.HYPER_REG_P] = float(np.float32(math.log(cfg.w_reg)))

        self._cconf = self._make_config()
        n_part = self.lib.irs_sgld_partials_doubles(ctypes.byref(self._cconf))
        self._partials = torch.zeros(max(int(n_part), 1), device=dev, dtype=torch.float64)
        # launch arguments and captured graphs exist per IMAGE SET: the input pipeline alternates between two resident sets of
        # (fixed, moving, mask, fixed-side LCC terms) so that committing an uploaded pair is a pointer swap, not a copy
        self._set = 0
        self._cbufs = [None, None]
        self._graph_sets = [{}, {}]   # per set: transitions per replay -> captured CUDA graph
        self.iteration = 0

        # posterior moments (Welford): displacement (3,V) and warped image (1,V)
        self.n_kept = 0
        self.disp_mean = torch.zeros(3, D, H, W, **f32)
        self.disp_m2 = torch.zeros(3, D, H, W, **f32)
        self.im_mean = torch.zeros(1, D, H, W, **f32)
        self.im_m2 = torch.zeros(1, D, H, W, **f32)

        self._lin = [torch.linspace(-1, 1, steps=n).to(dev) for n in (W, H, D)]  # utils/util.py:270-272 of the reference

        # split-R-hat accumulators (enable_convergence_diagnostics): None while disabled
        self._rhat = None
        # label counts of the segmentation posterior (enable_segmentation_posterior): None while disabled
        self._segpost = None
        # accumulators of the Jacobian posterior (enable_jacobian_posterior): None while disabled
        self._jacpost = None
        # landmark pairs and accumulators of the landmark posterior (enable_landmark_posterior): None while disabled
        self._lmpost = None

    # ------------------------------------------------------------------------------------------------------------------
    def _make_config(self):
        cfg = self.cfg
        c = _lib.SgldConfig()
        c.C, (c.D, c.H, c.W) = self.C, self.dims
        c.chain_offset = self.chain_offset
        c.data_term = _lib.DATA_LCC if cfg.data_loss == 'lcc' else _lib.DATA_SSD
        c.K, c.lcc_s = cfg.no_components, cfg.s
        c.reg_type = _lib.REG_LOGNORMAL if cfg.reg_loss == 'RegLoss_LogNormal' else _lib.REG_L2
        c.reg_learnable = int(cfg.reg_learnable)
        if cfg.sobolev_enabled:
            taps, _ = Sobolev_kernel_1D(cfg.sobolev_s, cfg.sobolev_lambda)
            taps = taps.astype(np.float32)  # `.float()` in trainer/trainer.py:573
            c.n_taps = len(taps)
            for i, t in enumerate(taps):
                c.taps[i] = float(t)
        else:
            c.n_taps = 0
        c.svf_steps = cfg.svf_steps
        c.virtual_decimation = int(cfg.virtual_decimation)
        c.use_jitter = int(cfg.uniform_noise)
        c.gather_radius_max = cfg.gather_radius_max
        c.hyper_mode = _lib.HYPER_MODES[cfg.hyper_mode]
        c.tau, c.jitter_alpha, c.w_reg, c.dof = cfg.tau, cfg.uniform_noise_magnitude, cfg.w_reg, self.dof
        c.lr_log_std, c.lr_logits, c.lr_reg0, c.lr_reg1 = cfg.lr_log_std, cfg.lr_logits, cfg.lr_reg, cfg.lr_reg
        c.lr_decay, (c.beta1, c.beta2), c.adam_eps = cfg.lr_decay, cfg.betas, cfg.adam_eps
        c.gmm_scale_prior_loc, c.gmm_scale_prior_scale = cfg.gmm_scale_prior
        c.dirichlet_alpha = cfg.dirichlet_alpha
        c.reg_scale_prior_loc, c.reg_scale_prior_scale = cfg.reg_scale_prior
        shape = 0.5 * self.dof  # parse_config.py:139-143 of the reference
        c.w_reg_prior_shape, c.w_reg_prior_rate = shape, 1.0 / shape
        c.n_mask = self.n_mask
        c.seed = cfg.seed
        if self.ffd:
            for a in range(3):
                c.ffd_cps[a], c.ffd_grid[a] = cfg.cps[a], self.state_dims[a]
                for j, k in enumerate(self._ffd_taps[a]):
                    c.ffd_kernel[a][j] = k
        return c

    def _buffers(self):
        b = _lib.SgldBuffers()
        p = lambda t: None if t is None else t.data_ptr()
        b.v, b.sigma = p(self.v), p(self.sigma)
        gD, gH, gW = self.state_dims
        b.sigma_chain_stride = 0 if self.sigma is None or self.sigma.shape[0] == 1 else 3 * gD * gH * gW
        b.fixed, b.moving, b.mask = p(self.fixed_term), p(self.moving_im), p(self.mask)
        b.eps, b.jitter_unit = p(self.eps_inject), p(self.jitter_inject)
        b.css, b.hist, b.im_warped, b.z = p(self.css), p(self.hist), p(self.im_warped), p(self.z)
        b.lcc_a, b.lcc_rs, b.scratch1, b.scratch2 = p(self._lcc_a), p(self._lcc_rs), p(self._scratch1), p(self._scratch2)
        b.field_a, b.field_b, b.grad_v = p(self._field_a), p(self._field_b), p(self.grad_v)
        b.maxabs, b.hyper, b.stats = p(self._maxabs), p(self.hyper), p(self.stats)
        b.gmm_table, b.partials, b.counters = p(self._gmm_table), p(self._partials), p(self._counters)
        if self.ffd:
            b.ffd_dense, b.ffd_grad = p(self._ffd_dense), p(self._ffd_grad)
            b.ffd_scratch, b.ffd_work = p(self._ffd_scratch), p(self._ffd_work)
        return b

    @property
    def _cbuf(self):
        return self._cbufs[self._set]

    @_cbuf.setter
    def _cbuf(self, value):
        self._cbufs[self._set] = value

    @property
    def _graphs(self):
        return self._graph_sets[self._set]

    def _invalidate(self):
        self._cbufs, self._graph_sets = [None, None], [{}, {}]

    # ------------------------------------------------------------------------------------------------------------------
    # initialisation (reference trainer/trainer.py:529-547, 585-611)
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def init_chains(self, MCMC_init='VI', var_params_q_v=None, generator=None, no_chains_total=None):
        """Trainer.__SGLD_init (reference trainer/trainer.py:585-611): 'VI' draws v_c = mu + eps_c sigma + x_c u (one
        sample_q_v call per chain, utils/sampler.py:4-21) and uses sigma = exp(log_var / 2) as the preconditioner;
        'identity' / 'noise' start from 0 / N(0,1) with sigma = 1.

        The draws follow the reference's order over GLOBAL chain ids: this shard (chains chain_offset .. chain_offset + C of
        no_chains_total) skips the numbers of the chains before it, so identically seeded ranks start every chain exactly
        where a single-GPU run with all chains would -- and no two shards start from the same states."""
        from .utils.sampler import draw_chain_states
        v, sigma = draw_chain_states(MCMC_init, var_params_q_v, self.C, self.chain_offset, no_chains_total, generator,
                                     state_shape=tuple(self.v.shape[1:]), device=self.device)
        self.v.copy_(v)
        self.sigma = sigma
        self._invalidate()

    @torch.no_grad()
    def set_state(self, v, sigma=None):
        self.v.copy_(v.to(self.device))
        self.sigma = None if sigma is None else sigma.to(self.device, torch.float32).contiguous()
        if self.sigma is not None and self.sigma.shape[0] not in (1, self.C):
            raise ValueError('sigma must have 1 or no_chains entries in dim 0')
        self._invalidate()

    @torch.no_grad()
    def init_gmm(self, v_sample=None, warm_up=25, sigma_hat=None):
        """Trainer.__GMM_init: sigma_hat from one un-noised forward pass, log_std = linspace(log s/100, log 5s, K),
        then `warm_up` Adam steps.  `sigma_hat` given: only GMM.init_parameters (model/loss.py:61-65)."""
        K = self.cfg.no_components
        if sigma_hat is not None:
            if self.cfg.data_loss == 'ssd':   # one Gaussian at the residuals' own scale (see SSD.init_parameters)
                ls = torch.full((K,), math.log(sigma_hat))
            else:
                ls = torch.linspace(math.log(sigma_hat / 100.0), math.log(sigma_hat * 5.0), steps=K)
            self.hyper[..., _lib.HYPER_LOG_STD:_lib.HYPER_LOG_STD + K] = ls.double().to(self.device)
            return
        if v_sample is None:
            v_sample = self.v[:1]
        v_sample = v_sample.to(self.device, torch.float32).contiguous()
        b = self._buffers()
        _lib.check(self.lib.irs_sgld_gmm_init(ctypes.byref(self._cconf), ctypes.byref(b), _lib.ptr(v_sample), warm_up,
                                              _lib.stream()))
        if self.per_chain:   # every chain starts from the same initialised mixture (and its warm-up Adam state)
            self.hyper[1:] = self.hyper[0]

    # ------------------------------------------------------------------------------------------------------------------
    # checkpoint / resume (SURVEY section 5: the reference has none -- a run that dies starts over)
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def state_dict(self):
        """everything the chains carry between transitions, as host tensors: states, preconditioner, the shared mixture /
        regulariser parameters with their Adam moments and the Philox offset (`hyper`), the running posterior moments.
        A sampler restored from it continues bit-identically (the noise is a function of seed, chain, iteration)."""
        sd = {'dims': tuple(self.dims), 'state_dims': tuple(self.state_dims), 'no_chains': self.C,
              'chain_offset': self.chain_offset, 'seed': self.cfg.seed, 'iteration': self.iteration,
              'v': self.v.cpu(), 'sigma': None if self.sigma is None else self.sigma.cpu(), 'hyper': self.hyper.cpu(),
              'n_kept': self.n_kept, 'disp_mean': self.disp_mean.cpu(), 'disp_m2': self.disp_m2.cpu(),
              'im_mean': self.im_mean.cpu(), 'im_m2': self.im_m2.cpu()}
        if self._rhat is not None:   # convergence diagnostics enabled: their accumulators travel too
            r = self._rhat
            sd['rhat'] = {'N': r['N'], 'k': r['k'], 'mean': r['mean'].cpu(), 'm2': r['m2'].cpu()}
        if self._segpost is not None:   # segmentation posterior enabled: its label counts travel too
            p = self._segpost
            sd['segpost'] = {'labels': list(p['labels']), 'n': p['n'], 'counts': p['counts'].cpu()}
        if self._jacpost is not None:   # Jacobian posterior enabled: its accumulators travel too
            j = self._jacpost
            sd['jacpost'] = {'n': j['n'], 'folds': j['folds'].cpu(), 'mean': j['mean'].cpu(), 'm2': j['m2'].cpu()}
        if self._lmpost is not None:   # landmark posterior enabled: the landmarks, spacing and accumulators travel too
            lm = self._lmpost
            sd['lmpost'] = {'fixed': lm['fixed_host'].clone(), 'moving': lm['moving_host'].clone(), 'spacing': list(lm['spacing']),
                            'n': lm['n'], 'acc': lm['acc'].cpu()}
        return sd

    @torch.no_grad()
    def load_state_dict(self, sd):
        for key, mine in (('dims', tuple(self.dims)), ('state_dims', tuple(self.state_dims)), ('no_chains', self.C),
                          ('chain_offset', self.chain_offset), ('seed', self.cfg.seed)):
            if tuple(sd[key]) != mine if isinstance(mine, tuple) else sd[key] != mine:
                raise ValueError(f'checkpoint does not match this sampler: {key} = {sd[key]} (here {mine})')
        self.set_state(sd['v'], sd['sigma'])
        self.hyper.copy_(sd['hyper'])
        self.iteration, self.n_kept = int(sd['iteration']), int(sd['n_kept'])
        for name in ('disp_mean', 'disp_m2', 'im_mean', 'im_m2'):
            getattr(self, name).copy_(sd[name])
        # a checkpoint with diagnostics enables them here; one without leaves disabled diagnostics disabled and restarts
        # enabled ones from zero kept samples
        if 'rhat' in sd:
            self.enable_convergence_diagnostics(sd['rhat']['N'])
            self._rhat['k'] = int(sd['rhat']['k'])
            self._rhat['mean'].copy_(sd['rhat']['mean'])
            self._rhat['m2'].copy_(sd['rhat']['m2'])
        elif self._rhat is not None:
            self.enable_convergence_diagnostics(self._rhat['N'])
        # the same for the segmentation posterior: enabled with the checkpoint's labels and counts, or restarted from zero
        if 'segpost' in sd:
            self.enable_segmentation_posterior(sd['segpost']['labels'])
            self._segpost['n'] = int(sd['segpost']['n'])
            self._segpost['counts'].copy_(sd['segpost']['counts'])
        elif self._segpost is not None:
            self.enable_segmentation_posterior(self._segpost['labels'])
        # and for the Jacobian posterior
        if 'jacpost' in sd:
            self.enable_jacobian_posterior()
            self._jacpost['n'] = int(sd['jacpost']['n'])
            for name in ('folds', 'mean', 'm2'):
                self._jacpost[name].copy_(sd['jacpost'][name])
        elif self._jacpost is not None:
            self.enable_jacobian_posterior()
        # and for the landmark posterior (with the checkpoint's landmarks and spacing)
        if 'lmpost' in sd:
            lm = sd['lmpost']
            self.enable_landmark_posterior(lm['fixed'], lm['moving'], lm['spacing'])
            self._lmpost['n'] = int(lm['n'])
            self._lmpost['acc'].copy_(lm['acc'])
        elif self._lmpost is not None:
            lm = self._lmpost
            self.enable_landmark_posterior(lm['fixed_host'], lm['moving_host'], lm['spacing'])

    def set_noise(self, eps=None, jitter_unit=None):
        """explicit N(0,1) / U[0,1) numbers (C,3,D,H,W) instead of Philox: exact noise-on parity tests"""
        self.eps_inject = None if eps is None else eps.to(self.device, torch.float32).contiguous()
        self.jitter_inject = None if jitter_unit is None else jitter_unit.to(self.device, torch.float32).contiguous()
        self._invalidate()

    # ------------------------------------------------------------------------------------------------------------------
    # the transition
    # ------------------------------------------------------------------------------------------------------------------
    def launches_per_step(self):
        return int(self.lib.irs_sgld_launches_per_step(ctypes.byref(self._cconf)))

    def _enqueue(self):
        if self._cbuf is None:
            self._cbuf = self._buffers()
        _lib.check(self.lib.irs_sgld_step(ctypes.byref(self._cconf), ctypes.byref(self._cbuf), _lib.stream()))

    def capture(self, iters_per_graph=1):
        """capture `iters_per_graph` transitions into one CUDA graph (all state lives in device memory, so a replay needs no
        host work at all: a long run is a handful of graph launches).  Several graphs of different lengths may coexist;
        step() replays the longest one that still fits."""
        k = int(iters_per_graph)
        if k < 1:
            raise ValueError('iters_per_graph must be >= 1')
        if k in self._graphs:
            return
        self._enqueue()  # warm-up outside capture (function attributes, lazy module load)
        torch.cuda.synchronize()
        self.iteration += 1
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(k):
                self._enqueue()
        self._graphs[k] = g

    def step(self, n=1, use_graph=True):
        """run n transitions; asynchronous"""
        if use_graph and not self._graphs:
            self.capture()      # runs one transition itself
            n -= 1
        done = 0
        if use_graph:
            for k in sorted(self._graphs, reverse=True):
                while n - done >= k:
                    self._graphs[k].replay()
                    done += k
        while done < n:
            self._enqueue()
            done += 1
        self.iteration += max(n, 0)

    STAGES = ('langevin+sobolev', 'svf_fwd', 'reg_energy', 'warp', 'residual_map', 'mixture_step', 'dL/dz',
              'map+warp_adjoint', 'reg_hyper', 'svf_adjoint', 'reg_grad+update')

    def profile_stages(self):
        """one eager transition with CUDA events between the stages -> {stage: milliseconds} (synchronises)"""
        if self._cbuf is None:
            self._cbuf = self._buffers()
        ms = (ctypes.c_float * len(self.STAGES))()
        _lib.check(self.lib.irs_sgld_step_profile(ctypes.byref(self._cconf), ctypes.byref(self._cbuf), _lib.stream(), ms))
        self.iteration += 1
        return dict(zip(self.STAGES, [float(x) for x in ms]))

    @torch.no_grad()
    def load_images(self, fixed_im, moving_im, mask):
        """(re)load the image pair from host (pinned) or device tensors into the sampler's resident buffers; the
        fixed-image side of the LCC map is recomputed.  Buffer addresses do not change, so a captured graph stays valid."""
        self.fixed_im.copy_(fixed_im, non_blocking=True)
        self.moving_im.copy_(moving_im, non_blocking=True)
        self.mask.copy_(mask.view(torch.uint8) if mask.dtype == torch.bool else mask, non_blocking=True)
        if self.cfg.data_loss == 'lcc':
            D, H, W = self.dims
            _lib.check(self.lib.irs_lcc_normalise(_lib.ptr(self.fixed_im), self.cfg.s, _lib.ptr(self._lcc_a), None,
                                                  _lib.ptr(self.fixed_term), 1, D, H, W, _lib.stream()))

    @torch.no_grad()
    def prefetch_images(self, fixed_im, moving_im, mask):
        """Start uploading the NEXT image pair from (pinned) host memory into staging buffers on a dedicated copy stream
        and return immediately: the transfer -- and the fixed-image side of the LCC map, computed on the same stream once
        the fixed image has arrived -- overlap the transitions running on the compute stream.  The host tensors must stay
        unchanged until commit_images() has been called.  Double-buffered input pipeline of the sampler."""
        lcc = self.cfg.data_loss == 'lcc'
        if getattr(self, '_stage', None) is None:
            self._stage = (torch.empty_like(self.fixed_im), torch.empty_like(self.moving_im), torch.empty_like(self.mask))
            self._stage_term = torch.empty_like(self.fixed_term) if lcc else None
            self._stage_a = torch.empty_like(self.fixed_term) if lcc else None
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._stage_ready, self._stage_free = torch.cuda.Event(), torch.cuda.Event()
        cs = self._copy_stream
        cs.wait_event(self._stage_free)   # the previous commit has read the staging buffers (no-op before the first one)
        with torch.cuda.stream(cs):
            self._stage[0].copy_(fixed_im, non_blocking=True)
            if lcc:
                D, H, W = self.dims
                _lib.check(self.lib.irs_lcc_normalise(_lib.ptr(self._stage[0]), self.cfg.s, _lib.ptr(self._stage_a), None,
                                                      _lib.ptr(self._stage_term), 1, D, H, W, _lib.stream()))
            self._stage[1].copy_(moving_im, non_blocking=True)
            self._stage[2].copy_(mask.view(torch.uint8) if mask.dtype == torch.bool else mask, non_blocking=True)
            self._stage_ready.record(cs)

    @torch.no_grad()
    def commit_images(self, swap=True):
        """Make the pair uploaded by prefetch_images() the current one.  swap (default): the staging buffers BECOME the
        resident set and the old resident set becomes the next staging area -- no device-to-device copies; launch
        arguments and CUDA graphs are kept per set (the first transition on a set captures its graph).  swap=False copies
        into the resident buffers instead (one set of graphs)."""
        if getattr(self, '_stage', None) is None:
            raise RuntimeError('commit_images() without a preceding prefetch_images()')
        cur = torch.cuda.current_stream()
        cur.wait_event(self._stage_ready)
        if swap:
            (self.fixed_im, self.moving_im, self.mask), self._stage = self._stage, (self.fixed_im, self.moving_im, self.mask)
            if self.cfg.data_loss == 'lcc':
                self.fixed_term, self._stage_term = self._stage_term, self.fixed_term
            else:
                self.fixed_term = self.fixed_im
            self._set ^= 1
        else:
            self.fixed_im.copy_(self._stage[0], non_blocking=True)
            self.moving_im.copy_(self._stage[1], non_blocking=True)
            self.mask.copy_(self._stage[2], non_blocking=True)
            if self.cfg.data_loss == 'lcc':
                self.fixed_term.copy_(self._stage_term, non_blocking=True)
        # the next prefetch overwrites what is now the staging set: it must wait for the transitions enqueued so far
        self._stage_free.record(cur)

    # ------------------------------------------------------------------------------------------------------------------
    # outputs of the last transition (views, no copies: SURVEY K13)
    # ------------------------------------------------------------------------------------------------------------------
    @property
    def displacement(self):
        return self.hist[-1]

    def transformation(self):
        T = torch.empty_like(self.displacement)
        D, H, W = self.dims
        _lib.check(self.lib.irs_svf_outputs(_lib.ptr(self.displacement), _lib.ptr(self._lin[0]), _lib.ptr(self._lin[1]),
                                            _lib.ptr(self._lin[2]), _lib.ptr(T), None, self.C, D, H, W, _lib.stream()))
        return T

    def output(self):
        """the reference's `output` dict (trainer/trainer.py:302-305) as views of the sampler's buffers"""
        return {'im_moving_warped': self.im_warped, 'displacement': self.displacement,
                'transformation': self.transformation(), 'curr_state': self.css}

    def loss_terms(self):
        """the reference's loss_terms / aux scalars (trainer/trainer.py:313-327); one device->host copy"""
        s = self.stats.cpu()
        return {'data': s[:, _lib.STAT_DATA].float(), 'reg': s[:, _lib.STAT_REG].float(),
                'alpha': s[:, _lib.STAT_ALPHA].float(), 'reg_energy': s[:, _lib.STAT_ENERGY].float()}

    def gmm_parameters(self):
        """(log_std, logits) of the mixture: (K,) each, or (C, K) with hyper_mode='per_chain'"""
        K = self.cfg.no_components
        h = self.hyper.cpu()
        return (h[..., _lib.HYPER_LOG_STD:_lib.HYPER_LOG_STD + K].float(),
                h[..., _lib.HYPER_LOGITS:_lib.HYPER_LOGITS + K].float())

    def reg_parameters(self):
        h = self.hyper.cpu()
        return h[..., _lib.HYPER_REG_P:_lib.HYPER_REG_P + 2]

    def warp_segmentation(self, seg=None, transformation=None):
        """nearest-neighbour warp of the moving segmentation with the current transformations (trainer.py:419)"""
        seg = self.moving_seg if seg is None else seg.to(self.device).contiguous()
        T = self.transformation() if transformation is None else transformation
        D, H, W = self.dims
        out = torch.empty(self.C, 1, D, H, W, device=self.device, dtype=seg.dtype)
        stride = 0 if seg.shape[0] == 1 else self.V
        if seg.dtype == torch.int16:
            fn = self.lib.irs_warp3d_nearest_i16
            _lib.check(fn(_lib.ptr(seg), stride, _lib.ptr(T), _lib.ptr(out), self.C, D, H, W, _lib.stream()))
        elif seg.dtype in (torch.bool, torch.uint8):
            fn = self.lib.irs_warp3d_nearest_u8
            _lib.check(fn(_lib.ptr(seg.view(torch.uint8)), stride, _lib.ptr(T), _lib.ptr(out.view(torch.uint8)), self.C,
                          D, H, W, _lib.stream()))
        else:
            raise NotImplementedError
        return out

    # ------------------------------------------------------------------------------------------------------------------
    # posterior moments
    # ------------------------------------------------------------------------------------------------------------------
    def accumulate(self, seg_warped=None, transformation=None):
        """fold the current sample of every chain into the running moments (kept-sample rule: trainer.py:414-430), when
        convergence diagnostics are enabled into the chain's split-R-hat sequence, and when the segmentation posterior is
        enabled the warped moving segmentation of every chain into its label counts: `seg_warped` (C,1,D,H,W) int16 if the
        caller has it already (warp_segmentation() of the current transformations), else warped here.  Without the
        segmentation posterior `seg_warped` is not used.  When the Jacobian posterior is enabled, log det J of every chain's
        transformation is folded into its accumulators and last_jacobian_stats is overwritten: `transformation` (C,3,D,H,W)
        fp32 if the caller has it already (transformation() of the current state), else computed here.  When the landmark
        posterior is enabled, the fixed landmarks are carried through the same transformation and folded into its
        accumulators, and last_landmark_stats is overwritten.  Without either `transformation` is not used."""
        n3, n1 = 3 * self.V, self.V
        st = _lib.stream()
        if self._rhat is not None and self._rhat['k'] >= self._rhat['N']:
            raise RuntimeError(f'convergence diagnostics were enabled for {self._rhat["N"]} kept samples per chain: this is '
                               f'sample {self._rhat["k"] + 1} (enable_convergence_diagnostics again to start over)')
        p = self._segpost
        if p is not None:
            if seg_warped is None:
                seg_warped = self.warp_segmentation()
            if seg_warped.dtype != torch.int16 or tuple(seg_warped.shape) != (self.C, 1, *self.dims) or \
                    not seg_warped.is_cuda or not seg_warped.is_contiguous():
                raise ValueError(f'seg_warped must be a contiguous ({self.C}, 1, {", ".join(map(str, self.dims))}) int16 '
                                 f'CUDA tensor')
        j, lm = self._jacpost, self._lmpost
        if j is not None or lm is not None:
            if transformation is None:
                transformation = self.transformation()
            if transformation.dtype != torch.float32 or tuple(transformation.shape) != (self.C, 3, *self.dims) or \
                    not transformation.is_cuda or not transformation.is_contiguous():
                raise ValueError(f'transformation must be a contiguous ({self.C}, 3, {", ".join(map(str, self.dims))}) fp32 '
                                 f'CUDA tensor')
        _lib.check(self.lib.irs_welford_update(_lib.ptr(self.displacement), self.C, n3, float(self.n_kept),
                                               _lib.ptr(self.disp_mean), _lib.ptr(self.disp_m2), st))
        _lib.check(self.lib.irs_welford_update(_lib.ptr(self.im_warped), self.C, n1, float(self.n_kept),
                                               _lib.ptr(self.im_mean), _lib.ptr(self.im_m2), st))
        self.n_kept += self.C
        r = self._rhat
        if r is not None:
            # kept sample k of N: the first floor(N/2) feed half 0, the last floor(N/2) half 1, the middle one of an odd N neither
            k, N, n = r['k'], r['N'], r['N'] // 2
            half, count = (0, k) if k < n else ((1, k - (N - n)) if k >= N - n else (None, None))
            if half is not None:
                _lib.check(self.lib.irs_split_welford_update(_lib.ptr(self.displacement), _lib.ptr(self.im_warped), self.C,
                                                             self.V, half, float(count), _lib.ptr(r['mean']),
                                                             _lib.ptr(r['m2']), st))
            r['k'] = k + 1
        if p is not None:
            _lib.check(self.lib.irs_label_counts_update(_lib.ptr(seg_warped), self.C, self.V, p['host_labels'],
                                                        len(p['labels']), _lib.ptr(p['counts']), st))
            p['n'] += self.C
        if j is not None:
            D, H, W = self.dims
            _lib.check(self.lib.irs_jacobian_update(_lib.ptr(transformation), _lib.ptr(self.mask), self.C, D, H, W,
                                                    float(j['n']), _lib.ptr(j['folds']), _lib.ptr(j['mean']),
                                                    _lib.ptr(j['m2']), _lib.ptr(j['stats']), _lib.ptr(j['partials']),
                                                    _lib.ptr(j['counters']), st))
            j['n'] += self.C
        if lm is not None:
            D, H, W = self.dims
            P = lm['P']
            _lib.check(self.lib.irs_landmark_map(_lib.ptr(transformation), self.C, D, H, W, _lib.ptr(lm['fixed']),
                                                 _lib.ptr(lm['moving']), P, lm['host_spacing'], _lib.ptr(lm['pred']),
                                                 _lib.ptr(lm['tre']), st))
            _lib.check(self.lib.irs_landmark_update(_lib.ptr(lm['pred']), _lib.ptr(lm['tre']), self.C, P, float(lm['n']),
                                                    _lib.ptr(lm['acc']), _lib.ptr(lm['stats']), st))
            lm['n'] += self.C

    def posterior_moments(self, group=None):
        """
        (mean, std) of the displacement and of the warped image over all kept samples of ALL ranks: the per-rank
        Welford triples are merged with Chan's formula through two all-reduces over NCCL (SURVEY section 8e).
        Returns a dict; std is unbiased like torch.std (utils/util.py:117).
        """
        from .parallel import merge_moments
        n, (dm, dm2), (im, im2) = merge_moments(self.n_kept, [(self.disp_mean, self.disp_m2), (self.im_mean, self.im_m2)],
                                                group)
        out = {'n': n, 'displacement_mean': dm, 'im_mean': im}
        for key, m2 in (('displacement_std', dm2), ('im_std', im2)):
            std = torch.full_like(m2, float('nan'))  # torch.std of fewer than two samples
            if n >= 2:
                _lib.check(self.lib.irs_welford_std(_lib.ptr(m2), float(n), _lib.ptr(std), m2.numel(), _lib.stream()))
            out[key] = std
        return out

    # ------------------------------------------------------------------------------------------------------------------
    # convergence diagnostics (voxel-wise split R-hat)
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def enable_convergence_diagnostics(self, n_kept_per_chain):
        """
        Allocate (or reset) the split-R-hat accumulators for the next `n_kept_per_chain` = N kept samples of every chain: a
        Welford (mean, M2) of the displacement (3,V) and the warped image (1,V) for the first and for the last floor(N/2)
        samples of each chain (the middle one of an odd N is dropped) -- 64 C V bytes of fp32, e.g. 8.6 GB for 64 chains at
        128^3.  accumulate() then also updates them (one launch, no synchronisation; the pooled moments are unchanged) and
        raises on sample N + 1; convergence_diagnostics() needs all N.
        With hyper_mode='reference' the chains share the mixture / regulariser parameters they step in turn, so they are not
        independent: R-hat is still computed, but its reading as a between-independent-chains check holds for 'per_chain' and
        'frozen'.
        """
        N = int(n_kept_per_chain)
        if N < 4:
            raise ValueError('split R-hat needs at least 4 kept samples per chain (2 draws in each half)')
        D, H, W = self.dims
        if self._rhat is None or self._rhat['N'] != N:
            self._rhat = None   # release the old pair first
            mean = torch.zeros(2, self.C, 4, D, H, W, device=self.device, dtype=torch.float32)
            self._rhat = {'N': N, 'k': 0, 'mean': mean, 'm2': torch.zeros_like(mean)}
        else:
            self._rhat['k'] = 0
            self._rhat['mean'].zero_()
            self._rhat['m2'].zero_()

    def disable_convergence_diagnostics(self):
        """free the split-R-hat accumulators; accumulate() goes back to the pooled moments alone"""
        self._rhat = None

    @property
    def diagnostics_enabled(self):
        return self._rhat is not None

    @torch.no_grad()
    def convergence_diagnostics(self, group=None):
        """
        Split R-hat (BDA3 section 11.4) over the kept samples of ALL chains of ALL ranks of `group` (two SUM all-reduces of
        fp64 partial sums when torch.distributed is initialised): M = 2 x total chains sequences of n = floor(N/2) draws.
        Returns {'displacement': (3,D,H,W), 'im': (1,D,H,W) fp32 device maps,
                 'mask': {'displacement': {...}, 'im': {...}} over the fixed mask with, per component, 'max' (list), 'n_above_1.01'
                         and 'n_above_1.1' (lists of voxel counts), 'n_voxels' (mask size),
                 'n': draws per sequence, 'M': number of sequences}.
        Raises unless enabled and all N kept samples have been accumulated.
        """
        r = self._rhat
        if r is None:
            raise RuntimeError('convergence diagnostics are not enabled (enable_convergence_diagnostics(N) before sampling)')
        if r['k'] < r['N']:
            raise RuntimeError(f'convergence diagnostics need all {r["N"]} kept samples per chain; {r["k"]} accumulated')
        from . import ops
        D, H, W = self.dims
        n = r['N'] // 2
        rhat, summary, M = ops.split_rhat(r['mean'].view(2 * self.C, 4, D, H, W), r['m2'].view(2 * self.C, 4, D, H, W), n,
                                          self.mask.view(D, H, W), group=group)
        s = summary.cpu()

        def part(rows):
            return {'max': [float(x) for x in s[rows, 0]], 'n_above_1.01': [int(x) for x in s[rows, 1]],
                    'n_above_1.1': [int(x) for x in s[rows, 2]], 'n_voxels': int(self.n_mask)}
        return {'displacement': rhat[:3], 'im': rhat[3:], 'mask': {'displacement': part(slice(0, 3)), 'im': part(slice(3, 4))},
                'n': n, 'M': M}

    # ------------------------------------------------------------------------------------------------------------------
    # posterior of the warped segmentation (per-voxel label histogram)
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def enable_segmentation_posterior(self, labels):
        """
        Allocate (or reset) the label counts of the segmentation posterior: (L, D, H, W) int32 for the L = len(labels) labels
        (1..32 distinct non-zero int16 values; every other value of the segmentation is the class "other") -- 4 L V bytes
        whatever the number of chains, e.g. 126 MB for 15 labels at 128^3, 1.0 GB at 256^3.  accumulate() then also adds the
        warped moving segmentation of every chain (one launch, no synchronisation; moments, split R-hat and chain states are
        unchanged) and segmentation_posterior() gives the label probabilities, the majority labels and the entropy.
        Needs a moving segmentation (int16).
        """
        if self.moving_seg is None:
            raise ValueError('the segmentation posterior needs a moving segmentation (moving["seg"])')
        if self.moving_seg.dtype != torch.int16:
            raise NotImplementedError('the segmentation posterior needs an int16 moving segmentation')
        labels = [int(x) for x in labels]
        if not 1 <= len(labels) <= 32 or len(set(labels)) != len(labels) or 0 in labels or \
                not all(-32768 <= x <= 32767 for x in labels):
            raise ValueError(f'the segmentation posterior takes 1..32 distinct non-zero int16 labels, got {labels}')
        p = self._segpost
        if p is None or p['labels'] != labels:
            self._segpost = None   # release the old counts first
            counts = torch.zeros(len(labels), *self.dims, device=self.device, dtype=torch.int32)
            self._segpost = {'labels': labels, 'host_labels': (ctypes.c_int * len(labels))(*labels), 'n': 0, 'counts': counts}
        else:
            p['n'] = 0
            p['counts'].zero_()

    def disable_segmentation_posterior(self):
        """free the label counts; accumulate() no longer touches the segmentations"""
        self._segpost = None

    @property
    def segmentation_posterior_enabled(self):
        return self._segpost is not None

    @torch.no_grad()
    def segmentation_posterior(self, seg_fixed=None, group=None):
        """
        The posterior of the warped moving segmentation over every segmentation accumulated by ALL ranks of `group` (one SUM
        all-reduce of the integer counts when torch.distributed is initialised, parallel.merge_label_counts; the local counts are
        kept, so sampling can continue).  seg_fixed: int16 (1,1,D,H,W) for the overlap sums, or None.
        Returns {'labels': list, 'n': number of segmentations (kept samples x chains),
                 'probability': (L,D,H,W) fp32, 'majority': (1,1,D,H,W) int16, 'entropy': (1,D,H,W) fp32 device tensors,
                 'summary': (L,3) int64 device tensor, per label: S = sum of the counts (S / n = expected volume in voxels),
                            O = the same inside seg_fixed == label (0 without seg_fixed; 2 O / (S + n |F|) = soft Dice),
                            U = voxels with 0 < count < n}  (ops.label_posterior).
        """
        from . import ops
        from .parallel import merge_label_counts
        p = self._segpost
        if p is None:
            raise RuntimeError('the segmentation posterior is not enabled (enable_segmentation_posterior(labels) before sampling)')
        n, counts = merge_label_counts(p['n'], p['counts'], group)
        if n < 1:
            raise RuntimeError('the segmentation posterior has no accumulated segmentation yet')
        if seg_fixed is not None:
            seg_fixed = seg_fixed.to(self.device).contiguous()
        prob, majority, entropy, summary = ops.label_posterior(counts, n, p['labels'], seg_fixed)
        return {'labels': list(p['labels']), 'n': n, 'probability': prob, 'majority': majority, 'entropy': entropy,
                'summary': summary}

    # ------------------------------------------------------------------------------------------------------------------
    # posterior of the Jacobian determinant (folding probability, mean and std of log det J)
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def enable_jacobian_posterior(self):
        """
        Allocate (or reset) the accumulators of the Jacobian posterior: per voxel the number of folded samples (int32) and
        the Welford mean / M2 (fp32) of log det J over the finite samples -- 12 V bytes whatever the number of chains, 25 MB
        at 128^3, 201 MB at 256^3.  accumulate() then also folds log det J of every chain's transformation into them (one
        launch, no synchronisation; moments, split R-hat, label counts and chain states are unchanged) and keeps the per-chain
        sums of that sample over the mask in last_jacobian_stats; jacobian_posterior() gives the maps and summaries.
        """
        j = self._jacpost
        if j is None:
            from . import ops
            partials, counters = ops.jacobian_scratch(self.C, self.device)
            z = dict(device=self.device, dtype=torch.float32)
            self._jacpost = {'n': 0, 'folds': torch.zeros(*self.dims, device=self.device, dtype=torch.int32),
                             'mean': torch.zeros(*self.dims, **z), 'm2': torch.zeros(*self.dims, **z),
                             'stats': torch.zeros(self.C, 4, device=self.device, dtype=torch.float64),
                             'partials': partials, 'counters': counters}
        else:
            j['n'] = 0
            for name in ('folds', 'mean', 'm2', 'stats'):
                j[name].zero_()

    def disable_jacobian_posterior(self):
        """free the accumulators; accumulate() no longer computes log det J"""
        self._jacpost = None

    @property
    def jacobian_posterior_enabled(self):
        return self._jacpost is not None

    @property
    def last_jacobian_stats(self):
        """(C,4) fp64 device tensor of the latest accumulated sample, per chain over the fixed mask: finite voxels, folded
        voxels, sum of log det J and of its square over the finite voxels (overwritten by every accumulate(); copy it to keep
        it).  The population std of log det J over the finite mask voxels, SDlogJ, is sqrt(s2 / n - (s / n)^2).  Registration
        challenges that report SDlogJ clip det J at 1e-9 instead of leaving the non-positive voxels out."""
        if self._jacpost is None:
            raise RuntimeError('the Jacobian posterior is not enabled (enable_jacobian_posterior() before sampling)')
        return self._jacpost['stats']

    @torch.no_grad()
    def jacobian_posterior(self, group=None):
        """
        The Jacobian posterior over every sample accumulated by ALL ranks of `group` (parallel.merge_jacobian_moments, two SUM
        all-reduces when torch.distributed is initialised; the local accumulators are kept, so sampling can continue).
        Returns {'n': samples (kept samples x chains), 'fold_probability', 'log_det_J_mean', 'log_det_J_std': (D,H,W) fp32
                 device maps (ops.jacobian_posterior: NaN mean where every sample folds, NaN std with fewer than two finite
                 samples), 'summary': the mask summary of ops.jacobian_posterior}.
        """
        from . import ops
        from .parallel import merge_jacobian_moments
        j = self._jacpost
        if j is None:
            raise RuntimeError('the Jacobian posterior is not enabled (enable_jacobian_posterior() before sampling)')
        n, folds, mean, m2 = merge_jacobian_moments(j['n'], j['folds'], j['mean'], j['m2'], group)
        if n < 1:
            raise RuntimeError('the Jacobian posterior has no accumulated sample yet')
        p_fold, mean_out, std_out, summary = ops.jacobian_posterior(folds, mean, m2, n, self.mask.view(self.dims))
        return {'n': n, 'fold_probability': p_fold, 'log_det_J_mean': mean_out, 'log_det_J_std': std_out, 'summary': summary}

    # ------------------------------------------------------------------------------------------------------------------
    # landmark registration error and landmark posterior
    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def enable_landmark_posterior(self, fixed_landmarks, moving_landmarks, spacing):
        """
        Allocate (or reset) the landmark posterior for P corresponding landmark pairs: (P,3) zero-based (x, y, z) voxel
        coordinates, row i of the fixed landmarks corresponding to row i of the moving ones (fixed ones finite and inside the
        volume, moving ones finite: checked here, once), spacing (x, y, z) in mm.  accumulate() then also carries every fixed
        landmark through every chain's transformation and folds the predicted moving position and its target registration
        error (TRE) into per-landmark fp64 accumulators -- 88 P bytes, plus 32 C P bytes of per-sample scratch -- in two
        launches with no synchronisation; moments, split R-hat, label counts, Jacobian accumulators and chain states are
        unchanged.  last_landmark_stats keeps the per-chain TRE sums of the latest sample; landmark_posterior() gives the
        per-landmark table.
        """
        from . import ops
        p, q = ops.check_landmarks(fixed_landmarks, moving_landmarks, self.dims)
        sp = ops.landmark_spacing(spacing)
        P = p.shape[0]
        dev = self.device
        f64 = dict(device=dev, dtype=torch.float64)
        self._lmpost = None   # release the old buffers first
        self._lmpost = {'P': P, 'fixed_host': p, 'moving_host': q, 'fixed': p.to(dev), 'moving': q.to(dev), 'spacing': sp,
                        'host_spacing': (ctypes.c_double * 3)(*sp), 'n': 0,
                        'acc': torch.zeros(P, _lib.LANDMARK_ACC, **f64), 'pred': torch.empty(self.C, P, 3, **f64),
                        'tre': torch.empty(self.C, P, **f64), 'stats': torch.zeros(self.C, 3, **f64)}

    def disable_landmark_posterior(self):
        """free the landmark buffers; accumulate() no longer reads the landmarks"""
        self._lmpost = None

    @property
    def landmark_posterior_enabled(self):
        return self._lmpost is not None

    @property
    def last_landmark_stats(self):
        """(C,3) fp64 device tensor of the latest accumulated sample, per chain over the landmarks in index order: sum of the
        TREs, sum of their squares, max TRE (mm; overwritten by every accumulate(); copy it to keep it).  The mean TRE of
        the sample is the first column over P."""
        if self._lmpost is None:
            raise RuntimeError('the landmark posterior is not enabled (enable_landmark_posterior(...) before sampling)')
        return self._lmpost['stats']

    @torch.no_grad()
    def landmark_posterior(self, group=None):
        """
        The landmark posterior over every sample accumulated by ALL ranks of `group` (parallel.merge_landmark_moments, two fp64
        SUM all-reduces when torch.distributed is initialised; the local accumulators are kept, so sampling can continue).
        Returns {'n': samples (kept samples x chains), 'table': the (P,16) fp64 device table of ops.landmark_posterior,
                 'fixed_landmarks', 'moving_landmarks': the (P,3) fp64 host tables, 'spacing': (x, y, z)}.
        """
        from . import ops
        from .parallel import merge_landmark_moments
        lm = self._lmpost
        if lm is None:
            raise RuntimeError('the landmark posterior is not enabled (enable_landmark_posterior(...) before sampling)')
        n, acc = merge_landmark_moments(lm['n'], lm['acc'], group)
        if n < 1:
            raise RuntimeError('the landmark posterior has no accumulated sample yet')
        table = ops.landmark_posterior(acc, n, lm['moving_host'], lm['spacing'])
        return {'n': n, 'table': table, 'fixed_landmarks': lm['fixed_host'].clone(), 'moving_landmarks': lm['moving_host'].clone(),
                'spacing': list(lm['spacing'])}
