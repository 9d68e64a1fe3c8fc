"""
Trainer -- the SGLD part of the reference's Trainer (reference trainer/trainer.py) on the fused CUDA step.

Kept from the reference: the method names and signatures on the hot path (`_SGLD_transition(fixed, moving, data_loss,
reg_loss) -> (loss_terms, output, aux)`, `_run_MCMC`, the chain / mixture initialisation), the attribute names read from
the `trainer` section of the JSON config (`no_chains`, `MCMC_init`, `no_iters_burn_in`, `no_samples_MCMC`,
`log_period_MCMC`, `uniform_noise`), the kept-sample rule and the folding guard.  Dropped (SURVEY.md section 2, out of
scope): TensorBoard, MetricTracker, SimpleITK surface distances, the data loader.  Kept samples and the posterior statistics can
be written as NIfTI-1 / legacy VTK (`save_dir`; irsgmcmc_b200/logger/writers.py).

What differs by design: one transition is one CUDA-graph replay with no host synchronisation; the per-iteration
`.item()` logging of the reference (trainer.py:391-412) is replaced by on-device statistics read back on request;
samples are folded into on-device Welford moments instead of a host buffer (trainer.py:365-366,428-430,458), and with
several ranks the chains are sharded and the moments merged with NCCL.
"""
import time

import numpy as np
import torch

from .. import _lib, parallel
from ..sampler import SGLDConfig, SGLDSampler
from ..utils.util import calc_DSC_GPU, calc_no_non_diffeomorphic_voxels


def sampler_config_from_json(config):
    """map the reference's JSON config (configs/*/config.json) onto SGLDConfig"""
    dl, reg = config['data_loss'], config['reg_loss']
    tr = config['trainer']
    sob = config.get('Sobolev_grad', {'enabled': False})
    opt_gmm = config.get('optimizer_GMM', {}).get('args', {})
    opt_reg = config.get('optimizer_reg', {}).get('args', {})
    kw = dict(
        data_loss='ssd' if dl['type'] == 'SSD' else 'lcc',
        no_components=dl['args'].get('no_components', 1), s=dl['args'].get('s', 2),
        reg_loss=reg['type'], w_reg=reg['args']['w_reg'], reg_learnable=reg['args'].get('learnable', False),
        sobolev_enabled=sob.get('enabled', False), sobolev_s=sob.get('s', 3), sobolev_lambda=sob.get('lambda', 0.5),
        tau=config['optimizer_SG_MCMC']['args']['lr'],
        uniform_noise=tr['uniform_noise']['enabled'], uniform_noise_magnitude=tr['uniform_noise'].get('magnitude', 0.1),
        virtual_decimation=config.get('virtual_decimation', True),
        lr_log_std=opt_gmm.get('lr_log_std', 0.2), lr_logits=opt_gmm.get('lr_logits', 0.2),
        lr_reg=opt_reg.get('lr_loc', opt_reg.get('lr_log_w_reg', 0.01)), lr_decay=opt_gmm.get('lr_decay', 1e-3))
    if 'data_loss_scale_prior' in config:
        a = config['data_loss_scale_prior']['args']
        kw['gmm_scale_prior'] = (a['loc'], a['scale'])
    if 'data_loss_proportion_prior' in config:
        kw['dirichlet_alpha'] = config['data_loss_proportion_prior']['args'].get('alpha', 0.5)
    if 'reg_loss_scale_prior' in config:
        a = config['reg_loss_scale_prior']['args']
        kw['reg_scale_prior'] = (a['loc'], a['scale'])
    if reg['type'] not in ('RegLoss_LogNormal', 'RegLoss_L2'):
        raise NotImplementedError(reg['type'])
    # "transformation_module": {"type": "SVF_3D" | "SVFFD_3D", "args": {"cps": [..]}} (configs/experiment5, parse_config.py:100-108)
    tm = config.get('transformation_module', {'type': 'SVF_3D', 'args': {}})
    if tm['type'] not in ('SVF_3D', 'SVFFD_3D'):
        raise NotImplementedError(tm['type'])
    kw['transformation'] = tm['type']
    # not a key of the reference: "trainer": {"hyper_mode": "reference" | "frozen" | "per_chain"} selects how the mixture / regulariser
    # hyper-parameters are stepped over the chains (SGLDConfig); the Trainer mirrors ONE parameter set into the drop-in modules, so
    # 'per_chain' is for the sampler API only
    kw['hyper_mode'] = tr.get('hyper_mode', 'reference')
    if kw['hyper_mode'] == 'per_chain':
        raise NotImplementedError("Trainer mirrors one shared parameter set: use SGLDSampler(SGLDConfig(hyper_mode='per_chain')) directly")
    if tm['type'] == 'SVFFD_3D':
        kw['cps'] = tm.get('args', {}).get('cps')
    return SGLDConfig(**kw)


class Trainer:
    def __init__(self, config, fixed, moving, var_params_q_v=None, structures_dict=None, device=None,
                 chain_offset=None, logger=None, save_dir=None, im_spacing=(1.0, 1.0, 1.0), sampler_config=None):
        """
        config: the reference's JSON config as a dict;  fixed / moving: {'im','mask','seg'} with shape (1,1,D,H,W)
        With torch.distributed initialised, `no_chains` is the TOTAL number of chains; this rank owns a contiguous shard.
        sampler_config: an SGLDConfig used instead of the one derived from `config`, e.g. with hyper_mode='per_chain' for
        independent chains.  The drop-in modules mirror ONE parameter set, so with 'per_chain' the Trainer runs without them
        (_run_MCMC() / _SGLD_transition() with data_loss = reg_loss = None).
        """
        self.config = config
        tr = config['trainer']
        self.MCMC_init = tr['MCMC_init']
        self.no_chains_total = int(tr['no_chains'])
        self.no_samples_MCMC = int(tr['no_samples_MCMC'])
        self.no_iters_burn_in = int(tr['no_iters_burn_in'])
        self.log_period_MCMC = int(tr['log_period_MCMC'])
        self.add_noise_uniform = tr['uniform_noise']['enabled']
        self.alpha = tr['uniform_noise'].get('magnitude', 0.1)
        self.virutal_decimation = config.get('virtual_decimation', True)  # (sic) reference trainer/trainer.py:42
        self.Sobolev_grad = config.get('Sobolev_grad', {}).get('enabled', False)
        self.structures_dict = structures_dict or {}
        self.logger = logger
        # save_dir: kept samples and the posterior statistics are written there as .nii.gz / .vtk with the reference's file
        # names (logger/logger.py:215-238); None = nothing touches the disk
        self.save_dir, self.im_spacing = save_dir, im_spacing

        world = torch.distributed.get_world_size() if torch.distributed.is_available() and torch.distributed.is_initialized() else 1
        if self.no_chains_total < world:   # every rank sees the same numbers: all of them raise, nobody hangs in a collective
            raise ValueError(f'no_chains = {self.no_chains_total} is smaller than the number of ranks ({world}): '
                             f'every rank needs at least one chain')
        offset, count = parallel.chain_shard(self.no_chains_total)
        if chain_offset is not None:
            offset = chain_offset
        self.no_chains = count
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        self.device = device
        self.fixed, self.moving = fixed, moving
        self.var_params_q_v = var_params_q_v
        self.sampler = SGLDSampler(fixed, moving, self.no_chains, sampler_config or sampler_config_from_json(config),
                                   device=device, chain_offset=offset)
        self.dims = self.sampler.dims
        self.no_voxels = int(np.prod(self.dims))
        self.SGLD_params = None
        self.return_masked_residuals = False
        self.clone_outputs = False
        self._gmm_pushed = False

    # -- initialisation (reference trainer.py:529-547, 585-611) ----------------------------------------------------
    def _GMM_init(self, v_sample=None):
        if v_sample is None and self.var_params_q_v is not None:
            from ..utils.sampler import sample_q_v
            v_sample = sample_q_v({k: v.to(self.device) for k, v in self.var_params_q_v.items()})
        self.sampler.init_gmm(v_sample)
        self._gmm_pushed = True

    def _SGLD_init(self, var_params_q_v=None, generator=None):
        var_params_q_v = var_params_q_v or self.var_params_q_v
        self.sampler.init_chains(self.MCMC_init, var_params_q_v, generator=generator, no_chains_total=self.no_chains_total)
        self.SGLD_params = {'sigma': self.sampler.sigma, 'tau': self.sampler.cfg.tau}
        self.v_curr_state = self.sampler.v

    # -- parameter mirroring between the drop-in modules and the device-side hyper state -----------------------------
    # The reference creates optimizer_GMM / optimizer_reg ONCE (trainer.py:62-66) and they persist through __GMM_init
    # (25 steps), VI (two mixture steps per iteration) and MCMC: MCMC starts with the decayed rate lr / (1 + step lr_decay),
    # warm moments and bias corrections counted from step 0.  The device keeps the same state in `hyper`
    # (csrc/irs_hyper.cuh), so parameters AND optimiser state travel in both directions.
    def _reg_params(self, reg_loss):
        if hasattr(reg_loss, 'loc'):
            return [reg_loss.loc, reg_loss.log_scale]
        return [reg_loss.log_w_reg]

    def _push_adam(self, optimizer, params, step_slot, m_slots, v_slots, beta_slot, sampler=None):
        h = (sampler or self.sampler).hyper
        betas = optimizer.param_groups[0]['betas']
        step = t = 0
        for p, ms, vs in zip(params, m_slots, v_slots):
            st = optimizer.state.get(p, {})
            k = p.numel()
            if len(st) == 0:
                h[ms:ms + k] = 0.0
                h[vs:vs + k] = 0.0
                continue
            step, t = int(st['step']), int(st['step']) - int(st.get('reinit', 0))
            h[ms:ms + k] = st['exp_avg'].detach().double().reshape(-1).to(h.device)
            h[vs:vs + k] = st['exp_avg_sq'].detach().double().reshape(-1).to(h.device)
        h[step_slot] = float(step)
        h[beta_slot] = betas[0] ** t       # the device multiplies these running products by beta once per step
        h[beta_slot + 1] = betas[1] ** t

    def _pull_adam(self, optimizer, params, step_slot, m_slots, v_slots, sampler=None):
        h = (sampler or self.sampler).hyper.cpu()
        step = int(round(float(h[step_slot])))
        for p, ms, vs in zip(params, m_slots, v_slots):
            k = p.numel()
            st = optimizer.state[p]
            st['step'] = step
            st.setdefault('reinit', 0)
            st['exp_avg'] = h[ms:ms + k].to(p.dtype).view_as(p).to(p.device)
            st['exp_avg_sq'] = h[vs:vs + k].to(p.dtype).view_as(p).to(p.device)

    def _push_hyper(self, data_loss, reg_loss, optimizer_GMM=None, optimizer_reg=None, sampler=None):
        from .. import _lib as L
        s = sampler or self.sampler
        if s.per_chain:
            raise NotImplementedError("hyper_mode='per_chain' has a parameter set per chain: the drop-in modules cannot mirror it")
        K = s.cfg.no_components
        optimizer_GMM = optimizer_GMM if optimizer_GMM is not None else getattr(self, 'optimizer_GMM', None)
        optimizer_reg = optimizer_reg if optimizer_reg is not None else getattr(self, 'optimizer_reg', None)
        if data_loss is not None:
            s.hyper[L.HYPER_LOG_STD:L.HYPER_LOG_STD + K] = data_loss.log_std.detach().double().to(s.device)
            s.hyper[L.HYPER_LOGITS:L.HYPER_LOGITS + K] = data_loss.logits.detach().double().to(s.device)
            if optimizer_GMM is not None:
                self._push_adam(optimizer_GMM, [data_loss.log_std, data_loss.logits], L.HYPER_GMM_STEP,
                                [L.HYPER_M_LOG_STD, L.HYPER_M_LOGITS], [L.HYPER_V_LOG_STD, L.HYPER_V_LOGITS],
                                L.HYPER_GMM_BETA_POW, sampler=s)
        if reg_loss is not None:
            params = self._reg_params(reg_loss)
            for i, p in enumerate(params):
                s.hyper[L.HYPER_REG_P + i] = p.detach().double()
            if optimizer_reg is not None and getattr(reg_loss, 'learnable', False):
                self._push_adam(optimizer_reg, params, L.HYPER_REG_STEP, [L.HYPER_REG_M + i for i in range(len(params))],
                                [L.HYPER_REG_V + i for i in range(len(params))], L.HYPER_REG_BETA_POW, sampler=s)

    @torch.no_grad()
    def _pull_hyper(self, data_loss, reg_loss, optimizer_GMM=None, optimizer_reg=None, with_optimizers=True, sampler=None):
        """device state -> modules.  with_optimizers=False copies the parameters only (device-to-device, no host
        synchronisation: what _SGLD_transition does after every step); the optimiser state needs the step counters on the
        host and is mirrored at the end of _run_MCMC / on request"""
        from .. import _lib as L
        s = sampler or self.sampler
        if s.per_chain:
            raise NotImplementedError("hyper_mode='per_chain' has a parameter set per chain: the drop-in modules cannot mirror it")
        K = s.cfg.no_components
        if with_optimizers:
            optimizer_GMM = optimizer_GMM if optimizer_GMM is not None else getattr(self, 'optimizer_GMM', None)
            optimizer_reg = optimizer_reg if optimizer_reg is not None else getattr(self, 'optimizer_reg', None)
        else:
            optimizer_GMM = optimizer_reg = None
        if data_loss is not None:
            data_loss.log_std.copy_(s.hyper[L.HYPER_LOG_STD:L.HYPER_LOG_STD + K].to(data_loss.log_std.dtype))
            data_loss.logits.copy_(s.hyper[L.HYPER_LOGITS:L.HYPER_LOGITS + K].to(data_loss.logits.dtype))
            if optimizer_GMM is not None:
                self._pull_adam(optimizer_GMM, [data_loss.log_std, data_loss.logits], L.HYPER_GMM_STEP,
                                [L.HYPER_M_LOG_STD, L.HYPER_M_LOGITS], [L.HYPER_V_LOG_STD, L.HYPER_V_LOGITS], sampler=s)
        if reg_loss is not None:
            params = self._reg_params(reg_loss)
            for i, p in enumerate(params):
                p.copy_(s.hyper[L.HYPER_REG_P + i].to(p.dtype))
            if optimizer_reg is not None and getattr(reg_loss, 'learnable', False):
                self._pull_adam(optimizer_reg, params, L.HYPER_REG_STEP, [L.HYPER_REG_M + i for i in range(len(params))],
                                [L.HYPER_REG_V + i for i in range(len(params))], sampler=s)

    # -- VI warm start (reference trainer.py:79-223): fused device path, and the drop-in modules through autograd -------
    def _build_VI_modules(self):
        """the objects the reference's ConfigParser would create for VI from the JSON (parse_config.py:110-148,215-249)"""
        from .. import model as M
        from ..optimizers import Adam
        from ..utils import RegistrationModule, SVF_3D, SVFFD_3D, Sobolev_kernel_1D
        cfg, sc, dev = self.config, self.sampler.cfg, self.device
        n = self.dims
        dof = 3.0 * float(np.prod(n))
        data_loss = (M.SSD() if sc.data_loss == 'ssd' else M.GMM(sc.no_components, sc.s)).to(dev)
        reg_cls = getattr(M, sc.reg_loss)
        reg_loss = reg_cls(w_reg=sc.w_reg, diff_op='GradientOperator', dims=n, learnable=sc.reg_learnable).to(dev)
        mods = {'data_loss': data_loss, 'reg_loss': reg_loss, 'entropy_loss': M.EntropyMultivariateNormal(),
                'scale_prior': M.LogScaleNormalPrior(*sc.gmm_scale_prior).to(dev),
                'proportion_prior': M.DirichletPrior(sc.no_components, sc.dirichlet_alpha).to(dev),
                'transformation_module': (SVFFD_3D(n, sc.cps) if sc.transformation == 'SVFFD_3D'
                                          else SVF_3D(n, sc.svf_steps)).to(dev),
                'registration_module': RegistrationModule()}
        if sc.reg_learnable:
            if sc.reg_loss == 'RegLoss_LogNormal':
                mods['loc_prior'] = M.LogEnergyExpGammaPrior(sc.w_reg, dof).to(dev)
                mods['reg_scale_prior'] = M.LogScaleNormalPrior(*sc.reg_scale_prior).to(dev)
                mods['optimizer_reg'] = Adam([{'params': [reg_loss.loc], 'lr': sc.lr_reg},
                                              {'params': [reg_loss.log_scale], 'lr': sc.lr_reg}], lr_decay=sc.lr_decay)
            else:
                shape = 0.5 * dof
                mods['w_reg_prior'] = M.LogPrecisionExpGammaPrior(shape=shape, rate=1.0 / shape).to(dev)
                mods['optimizer_reg'] = Adam(reg_loss.parameters(), lr=sc.lr_reg, lr_decay=sc.lr_decay)
        mods['optimizer_GMM'] = Adam([{'params': [data_loss.log_std], 'lr': sc.lr_log_std},
                                      {'params': [data_loss.logits], 'lr': sc.lr_logits}], lr_decay=sc.lr_decay)
        if sc.sobolev_enabled:
            taps = torch.from_numpy(Sobolev_kernel_1D(sc.sobolev_s, sc.sobolev_lambda)[0]).float().unsqueeze(0)
            S3 = torch.stack((taps, taps, taps), 0).to(dev)
            mods['S'] = {'x': S3.unsqueeze(2).unsqueeze(2), 'y': S3.unsqueeze(2).unsqueeze(4), 'z': S3.unsqueeze(3).unsqueeze(4)}
            mods['padding'] = (sc.sobolev_s,) * 6
        return mods

    def _step_GMM(self, m, residuals, alpha=1.0):
        """reference trainer.py:68-77"""
        data_loss = m['data_loss']
        data_term = data_loss(residuals.detach()).sum() * alpha
        data_term = data_term - m['scale_prior'](data_loss.log_scales).sum() - m['proportion_prior'](data_loss.log_proportions).sum()
        m['optimizer_GMM'].zero_grad()
        data_term.backward()
        m['optimizer_GMM'].step()

    def _get_VD_factor(self, m, residuals, mask):
        """reference trainer.py:507-514"""
        from ..utils import calc_VD_factor, rescale_residuals
        if not self.virutal_decimation:
            return 1.0
        return calc_VD_factor(rescale_residuals(residuals.detach(), mask, m['data_loss']), mask)

    def _calc_sample_loss_VI(self, m, fixed, moving, var_params_q_v, v_sample_unsmoothed, jitter_unit=None):
        """reference trainer.py:79-117 (Trainer.__calc_sample_loss_VI)"""
        from ..utils import SobolevGrad, calc_no_non_diffeomorphic_voxels, transform_coordinates, add_noise_uniform_field
        data_loss, reg_loss = m['data_loss'], m['reg_loss']
        v_sample = SobolevGrad.apply(v_sample_unsmoothed, m['S'], m['padding']) if 'S' in m else v_sample_unsmoothed
        transformation, displacement = m['transformation_module'](v_sample)
        with torch.no_grad():
            no_folded, log_det_J = calc_no_non_diffeomorphic_voxels(transformation, reg_loss.diff_op)
        if self.add_noise_uniform:
            if jitter_unit is not None:   # explicit U[0,1) numbers: exact parity tests
                transformation = transformation + transform_coordinates(-2.0 * self.alpha * jitter_unit + self.alpha)
            else:
                transformation = add_noise_uniform_field(transformation, self.alpha)
        im_moving_warped = m['registration_module'](moving['im'], transformation)
        output = {'displacement': displacement, 'transformation': transformation, 'im_moving_warped': im_moving_warped,
                  'log_det_J': log_det_J}
        residuals = data_loss.map(fixed['im'], im_moving_warped)
        alpha = self._get_VD_factor(m, residuals, fixed['mask'])
        residuals_masked = residuals[fixed['mask']]
        self._step_GMM(m, residuals_masked, alpha)
        data_term = data_loss(residuals_masked).sum() * alpha
        reg_term, log_y = reg_loss(v_sample)
        reg_term = reg_term.sum()
        entropy_term = m['entropy_loss'](sample=v_sample_unsmoothed, mu=var_params_q_v['mu'],
                                         log_var=var_params_q_v['log_var'], u=var_params_q_v['u']).sum()
        aux = {'alpha': alpha, 'reg_energy': log_y.exp(), 'no_non_diffeomorphic_voxels': no_folded,
               'residuals': residuals_masked}
        loss_terms = {'data': data_term, 'reg': reg_term, 'entropy': entropy_term}
        if reg_loss.learnable:
            if reg_loss.__class__.__name__ == 'RegLoss_LogNormal':
                loss_terms['reg_loc_prior'] = m['loc_prior'](log_y).sum()
            else:
                loss_terms['w_reg_prior'] = m['w_reg_prior'](reg_loss.log_w_reg)
        return loss_terms, output, aux

    def _run_VI_fused(self, var_params_q_v=None, no_iters=None, modules=None, lr=None, noise=None, history=True):
        """_run_VI on the fused device path (irsgmcmc_b200/vi.py, csrc/irs_vi.cu): no autograd, no eager field arithmetic.
        `history=False` enqueues all iterations without a host synchronisation (CUDA-graph replays)."""
        from ..vi import VIWarmStart
        tr = self.config['trainer']
        no_iters = int(tr.get('no_iters_VI', 0)) if no_iters is None else no_iters
        var_params_q_v = var_params_q_v or self.var_params_q_v
        m = modules or self._build_VI_modules()
        a = self.config.get('optimizer_q_v', {}).get('args', {})
        lr = lr or {'mu': a.get('lr_mu', 0.01), 'log_var': a.get('lr_log_var', 0.01), 'u': a.get('lr_u', 0.01)}
        vi = VIWarmStart(self.fixed, self.moving, var_params_q_v, self.sampler.cfg, device=self.device, lr_mu=lr['mu'],
                         lr_log_var=lr['log_var'], lr_u=lr['u'], lr_decay=a.get('lr_decay', 1e-3))
        # the mixture / regulariser parameters and the optimiser state of the stage before (mixture initialisation)
        self._push_hyper(m['data_loss'], m['reg_loss'], m['optimizer_GMM'], m.get('optimizer_reg'), sampler=vi.sampler)
        hist = []
        if noise is None and not history:
            vi.step(no_iters)
        else:
            for it in range(no_iters):
                if noise is not None:
                    eps, x, j1, j2 = next(noise)
                    vi.set_noise(eps, x, None if j1 is None else torch.cat((j1, j2), 0))
                vi.step(1, use_graph=noise is None)
                if history:
                    lt = vi.loss_terms()
                    entropy = lt['entropy_sample'] + lt['entropy_log_det']
                    # `loss` without the hyper-prior constants of the eager path's history (they carry no field gradient)
                    hist.append({'data_samples': lt['data'], 'reg_samples': lt['reg'], 'alpha_samples': lt['alpha'],
                                 'entropy': entropy, 'alpha': lt['alpha'][0], 'data': lt['data'].mean(), 'reg': lt['reg'].mean(),
                                 'loss': lt['data'].mean() + lt['reg'].mean() - entropy})
        self._pull_hyper(m['data_loss'], m['reg_loss'], m['optimizer_GMM'], m.get('optimizer_reg'), sampler=vi.sampler)
        self.var_params_q_v = {k: v.detach().clone() for k, v in vi.var_params().items()}
        self._vi_modules, self._vi = m, vi
        self.optimizer_GMM, self.optimizer_reg = m['optimizer_GMM'], m.get('optimizer_reg')
        self._gmm_pushed = False
        return self.var_params_q_v, m, hist

    def _run_VI(self, var_params_q_v=None, no_iters=None, modules=None, lr=None, noise=None, fused=True):
        """
        fit the Gaussian variational posterior q(v) (reference trainer.py:119-223): per iteration two antithetic samples,
        loss = data + reg - entropy, Adam on (mu, log_var, u) and on the regulariser hyper-parameters; the shared mixture
        is stepped inside each sample's loss.  Returns (var_params_q_v, modules, history of loss terms).
        `fused` (default): the device path of _run_VI_fused; False: the drop-in modules through autograd (what a user of the
        reference's classes gets; also the check of the fused path).
        `noise`: optional iterator of (eps, x, jitter1, jitter2) for exact parity tests.
        """
        if fused:
            return self._run_VI_fused(var_params_q_v, no_iters, modules, lr, noise)
        from ..optimizers import Adam
        tr = self.config['trainer']
        no_iters = int(tr.get('no_iters_VI', 0)) if no_iters is None else no_iters
        var_params_q_v = var_params_q_v or self.var_params_q_v
        vp = {k: v.detach().clone().to(self.device).requires_grad_(True) for k, v in var_params_q_v.items()}
        m = modules or self._build_VI_modules()
        a = self.config.get('optimizer_q_v', {}).get('args', {})
        lr = lr or {'mu': a.get('lr_mu', 0.01), 'log_var': a.get('lr_log_var', 0.01), 'u': a.get('lr_u', 0.01)}
        optimizer_q_v = Adam([{'params': [vp[k]], 'lr': lr[k]} for k in ('mu', 'log_var', 'u')],
                             lr_decay=a.get('lr_decay', 1e-3))
        fixed = {k: v.to(self.device) for k, v in self.fixed.items()}
        moving = {k: v.to(self.device) for k, v in self.moving.items()}
        history = []
        for it in range(no_iters):
            sigma = torch.exp(0.5 * vp['log_var'])
            if noise is not None:
                eps, x, j1, j2 = next(noise)
            else:
                eps, x, j1, j2 = torch.randn_like(sigma), torch.randn(1, device=self.device), None, None
            delta = eps * sigma + x * vp['u']          # utils/sampler.py:4-21, antithetic pair
            lt1, output, aux = self._calc_sample_loss_VI(m, fixed, moving, vp, vp['mu'] + delta, j1)
            lt2, _, _ = self._calc_sample_loss_VI(m, fixed, moving, vp, vp['mu'] - delta, j2)
            data_loss, reg_loss = m['data_loss'], m['reg_loss']
            data_term = (lt1['data'] + lt2['data']) / 2.0
            data_term = data_term - m['scale_prior'](data_loss.log_scales).sum() - m['proportion_prior'](data_loss.log_proportions).sum()
            reg_term = (lt1['reg'] + lt2['reg']) / 2.0
            if reg_loss.learnable:
                if reg_loss.__class__.__name__ == 'RegLoss_LogNormal':
                    reg_term = reg_term - (lt1['reg_loc_prior'] + lt2['reg_loc_prior']) / 2.0 - m['reg_scale_prior'](reg_loss.log_scale).sum()
                else:
                    reg_term = reg_term - (lt1['w_reg_prior'] + lt2['w_reg_prior']) / 2.0
            entropy_term = (lt1['entropy'] + lt2['entropy']) / 2.0 + m['entropy_loss'](log_var=vp['log_var'], u=vp['u']).sum()
            loss = data_term + reg_term - entropy_term
            if reg_loss.learnable:
                m['optimizer_reg'].zero_grad()
            optimizer_q_v.zero_grad()
            loss.backward()
            if reg_loss.learnable:
                m['optimizer_reg'].step()
            optimizer_q_v.step()
            history.append({'data': data_term.detach(), 'reg': reg_term.detach(), 'entropy': entropy_term.detach(),
                            'loss': loss.detach(), 'alpha': aux['alpha'],
                            'data_samples': torch.stack((lt1['data'].detach(), lt2['data'].detach())),
                            'reg_samples': torch.stack((lt1['reg'].detach(), lt2['reg'].detach()))})
        self.var_params_q_v = {k: v.detach() for k, v in vp.items()}
        self._vi_modules, self._optimizer_q_v, self._vp_leaves = m, optimizer_q_v, vp
        # one optimiser per hyper-parameter group for the whole run (reference trainer.py:62-66): MCMC continues with them
        self.optimizer_GMM, self.optimizer_reg = m['optimizer_GMM'], m.get('optimizer_reg')
        self._gmm_pushed = False   # the next transition pushes the parameters AND the optimiser state VI left behind
        return self.var_params_q_v, m, history

    @torch.no_grad()
    def _test_VI(self, var_params_q_v=None, no_samples=None, modules=None, speed_test_samples=100, with_ASD=True,
                 with_seg_posterior=False, with_jacobian_posterior=False, with_HD=False, HD_percentile=95.0, with_TRE=False):
        """
        evaluation of the fitted q(v) (reference trainer.py:226-289): `no_samples_VI_test` draws from q(v) -> Sobolev smoothing ->
        transformation -> number of folded voxels + log det J, warped image and segmentation, ASD / DSC per structure, the sample on
        disk; then the registration at the posterior mean, the sample mean / standard deviation of the displacement, and the
        sampling speed test (draw + transformation + image and segmentation warps).  The reference keeps every displacement in a
        host buffer for torch.std; here they are folded into Welford moments on the device (same unbiased result).
        Returns {'no_non_diffeomorphic_voxels': [S], 'DSC': (S, structures), 'ASD': (S, structures) | str, 'mean', 'std_dev' (3,D,H,W),
        'displacement_mu', 'im_moving_warped_mu', 'samples_per_sec'}.
        with_seg_posterior=True (needs structures_dict, both segmentations and S >= 1, else ValueError) adds 'seg_posterior',
        the posterior of the warped moving segmentation over the S draws (n = S), with the entries of _run_MCMC's; with
        save_dir, VI_seg_majority.nii.gz and VI_seg_entropy.nii.gz.
        with_jacobian_posterior=True (S >= 1, else ValueError) adds 'jacobian_posterior', the posterior of log det J over the
        S draws with the entries of _run_MCMC's ('SDlogJ' and 'folded_fraction' are (S, 1)); with save_dir,
        VI_log_det_J_mean.nii.gz, VI_log_det_J_std_dev.nii.gz and VI_fold_probability.nii.gz.
        with_HD=True (needs the segmentations, like 'ASD') adds 'HD' and 'HD95' (the key follows HD_percentile: 'HD99' for 99),
        (S, structures) arrays of the Hausdorff distance and its percentile per draw (utils.util.calc_HD_GPU; with with_ASD, one
        distance transform gives all three); with with_seg_posterior, 'HD_majority' and 'HD95_majority' per structure.
        with_TRE=True (needs 'landmarks' in both the fixed and the moving dict with the same P, and S >= 1, else ValueError) adds
        'TRE' (S, 1), the mean target registration error of the landmarks per draw, and 'landmark_posterior' over the S draws
        with the entries of _run_MCMC's; with save_dir, VI_landmarks.vtk.
        """
        from .. import ops
        from ..utils import SobolevGrad, calc_metrics
        from ..utils.sampler import sample_q_v
        tr = self.config['trainer']
        S = int(tr.get('no_samples_VI_test', 0)) if no_samples is None else int(no_samples)
        m = modules or getattr(self, '_vi_modules', None) or self._build_VI_modules()
        dev = self.device
        vp = {k: v.detach().to(dev, torch.float32) for k, v in (var_params_q_v or self.var_params_q_v).items()}
        moving = {k: v.to(dev) for k, v in self.moving.items()}
        seg_fixed = self.fixed['seg'].to(dev) if 'seg' in self.fixed else None
        with_seg = bool(self.structures_dict) and seg_fixed is not None and 'seg' in moving
        if with_seg_posterior:
            if not with_seg or S < 1:
                raise ValueError('with_seg_posterior=True needs structures_dict, fixed and moving segmentations and at least '
                                 'one sample')
            seg_labels = [int(x) for x in self.structures_dict.values()]
            seg_counts = torch.zeros(len(seg_labels), *self.dims, device=dev, dtype=torch.int32)
        if with_jacobian_posterior:
            if S < 1:
                raise ValueError('with_jacobian_posterior=True needs at least one sample')
            jac = {'folds': torch.zeros(*self.dims, device=dev, dtype=torch.int32),
                   'mean': torch.zeros(*self.dims, device=dev), 'm2': torch.zeros(*self.dims, device=dev),
                   'mask': self.fixed['mask'].to(dev).view(*self.dims), 'scratch': ops.jacobian_scratch(1, dev)}
            jac_traces = torch.zeros(S, 1, 4, device=dev, dtype=torch.float64)
        if with_TRE:
            if S < 1:
                raise ValueError('with_TRE=True needs at least one sample')
            lm_p, lm_q = self._landmark_pair()
            lm_acc = torch.zeros(lm_p.shape[0], _lib.LANDMARK_ACC, device=dev, dtype=torch.float64)
            lm_traces = torch.zeros(S, 1, 3, device=dev, dtype=torch.float64)
        transformation_module, registration_module, diff_op = m['transformation_module'], m['registration_module'], m['reg_loss'].diff_op

        def register(v):
            v_smoothed = SobolevGrad.apply(v, m['S'], m['padding']) if 'S' in m else v
            transformation, displacement = transformation_module(v_smoothed)
            return transformation, displacement, registration_module(moving['im'], transformation)

        mean, m2, count = torch.zeros((3, *self.dims), device=dev), torch.zeros((3, *self.dims), device=dev), 0
        folded, dsc, asd, hd, hd_q = [], [], [], [], []
        for test_sample_no in range(1, S + 1):
            transformation, displacement, im_moving_warped = register(sample_q_v(vp, no_samples=1))
            count = ops.welford_update(displacement.contiguous(), count, mean, m2)
            n_folded, log_det_J = calc_no_non_diffeomorphic_voxels(transformation, diff_op)
            folded.append(int(n_folded[0]))
            if with_jacobian_posterior:
                jac_traces[test_sample_no - 1] = ops.jacobian_update(transformation.contiguous(), jac['mask'], test_sample_no - 1,
                                                                     jac['folds'], jac['mean'], jac['m2'], jac['scratch'])
            if with_TRE:
                pred, tre = ops.landmark_map(transformation.contiguous(), lm_p, lm_q, self.im_spacing)
                lm_traces[test_sample_no - 1] = ops.landmark_update(pred, tre, test_sample_no - 1, lm_acc)
            if with_seg:
                seg_moving_warped = registration_module(moving['seg'], transformation)
                if with_ASD and not with_HD:
                    ASD, DSC = calc_metrics(seg_fixed, seg_moving_warped, self.structures_dict, self.im_spacing)
                    asd.append(ASD[0])
                else:
                    DSC = calc_DSC_GPU(1, seg_fixed, seg_moving_warped, self.structures_dict)
                    if with_HD:
                        ASD, HD, HD_q = self._surface_distances(seg_fixed, seg_moving_warped, 1, with_ASD, HD_percentile)
                        if with_ASD:
                            asd.append(ASD[0])
                        hd.append(HD[0])
                        hd_q.append(HD_q[0])
                dsc.append(DSC[0])
                if with_seg_posterior:
                    ops.label_counts_update(seg_moving_warped.contiguous(), seg_labels, seg_counts)
            if self.save_dir is not None:
                from ..logger import save_sample
                save_sample(self.save_dir, self.im_spacing, test_sample_no, im_moving_warped, displacement, log_det_J, model='VI')
        # the registration at the mean of the approximate posterior (reference trainer.py:257-262)
        _, displacement_mu, im_moving_warped_mu = register(vp['mu'])
        std_dev = ops.welford_std(m2, count) if count > 1 else torch.full_like(m2, float('nan'))   # torch.std of one sample is NaN
        if self.save_dir is not None:
            from ..logger import save_displacement_mean_and_std_dev, save_variational_posterior_mean
            save_variational_posterior_mean(self.save_dir, self.im_spacing, im_moving_warped_mu, displacement_mu)
            if count > 0:
                save_displacement_mean_and_std_dev(self.save_dir, self.im_spacing, mean, std_dev, moving.get('mask'), 'VI')
        result = {'no_non_diffeomorphic_voxels': folded, 'DSC': np.asarray(dsc), 'mean': mean, 'std_dev': std_dev,
                  'ASD': np.asarray(asd) if (with_seg and with_ASD) else 'unavailable: no segmentations / structures, or with_ASD=False',
                  'displacement_mu': displacement_mu, 'im_moving_warped_mu': im_moving_warped_mu, 'n': count}
        if with_HD:
            result.update(self._HD_entries(np.asarray(hd), np.asarray(hd_q), with_seg, HD_percentile))
        if with_seg_posterior:
            prob, majority, entropy, summary = ops.label_posterior(seg_counts, S, seg_labels, seg_fixed.contiguous())
            post = {'labels': seg_labels, 'n': S, 'probability': prob, 'majority': majority, 'entropy': entropy,
                    'summary': summary}
            result['seg_posterior'] = self._seg_posterior(post, with_ASD, 'VI', with_HD, HD_percentile)
        if with_jacobian_posterior:
            p_fold, mean_ld, std_ld, summary = ops.jacobian_posterior(jac['folds'], jac['mean'], jac['m2'], S, jac['mask'])
            post = {'n': S, 'fold_probability': p_fold, 'log_det_J_mean': mean_ld, 'log_det_J_std': std_ld, 'summary': summary}
            result['jacobian_posterior'] = self._jacobian_posterior(post, jac_traces, 'VI', gather=False)
        if with_TRE:
            post = {'n': S, 'table': ops.landmark_posterior(lm_acc, S, lm_q, self.im_spacing), 'fixed_landmarks': lm_p,
                    'moving_landmarks': lm_q, 'spacing': ops.landmark_spacing(self.im_spacing)}
            result['TRE'], result['landmark_posterior'] = self._landmark_posterior(post, lm_traces, 'VI', gather=False)
        if speed_test_samples:   # reference trainer.py:275-289
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(speed_test_samples):
                transformation, _, _ = register(sample_q_v(vp, no_samples=1))
                if 'seg' in moving:
                    registration_module(moving['seg'], transformation)
            torch.cuda.synchronize()
            result['samples_per_sec'] = speed_test_samples / (time.perf_counter() - t0)
        return result

    def _run_model(self, VI=None, MCMC=None, speed_test_iters=0):
        """the reference's Trainer._run_model (trainer.py:478-504): mixture initialisation (25 Adam steps), VI warm start,
        then SGLD -- with the mixture / regulariser parameters and their Adam state handed from stage to stage"""
        tr = self.config['trainer']
        VI = bool(tr.get('VI', False)) if VI is None else VI
        MCMC = bool(tr.get('MCMC', True)) if MCMC is None else MCMC
        self._GMM_init()
        m = self._build_VI_modules()
        self._pull_hyper(m['data_loss'], m['reg_loss'], m['optimizer_GMM'], m.get('optimizer_reg'))
        self.optimizer_GMM, self.optimizer_reg = m['optimizer_GMM'], m.get('optimizer_reg')
        result = {'modules': m}
        if VI:
            result['var_params_q_v'], _, result['VI_history'] = self._run_VI(modules=m)
            if int(tr.get('no_samples_VI_test', 0)) > 0:   # reference trainer.py:488-498: fit q(v), then sample from it
                result['VI_test'] = self._test_VI(modules=m, speed_test_samples=speed_test_iters)
        if MCMC:
            self._SGLD_init()
            self._gmm_pushed = False
            result.update(self._run_MCMC(m['data_loss'], m['reg_loss'], speed_test_iters=speed_test_iters))
        return result

    # -- the hot path -------------------------------------------------------------------------------------------------
    def _SGLD_transition(self, fixed=None, moving=None, data_loss=None, reg_loss=None):
        """
        one SGLD transition of every chain on this GPU; same return structure as the reference (trainer.py:291-356):
          loss_terms {'data': [C], 'reg': [C]},
          output {'im_moving_warped', 'displacement', 'transformation', 'curr_state'},
          aux {'residuals', 'alpha': [C], 'reg_energy': [C]}
        Scalars are returned as device tensors (no host synchronisation).  `data_loss` / `reg_loss`, when given, are
        the drop-in GMM / RegLoss modules: their parameters are pushed to the device state before the first transition
        and refreshed after every transition.
        """
        s = self.sampler
        if not self._gmm_pushed and (data_loss is not None or reg_loss is not None):
            self._push_hyper(data_loss, reg_loss)
            self._gmm_pushed = True
        s.step(1)
        if data_loss is not None or reg_loss is not None:
            self._pull_hyper(data_loss, reg_loss, with_optimizers=False)
        st = s.stats
        C = self.no_chains
        loss_terms = {'data': [st[c, 1].float() for c in range(C)], 'reg': [st[c, 2].float() for c in range(C)]}
        out = s.output()
        if self.clone_outputs:
            out = {k: v.detach().clone() for k, v in out.items()}
        residuals = s.z
        if self.return_masked_residuals:
            residuals = s.z[s.mask.bool().expand(C, -1, -1, -1, -1)].view(C, -1)
        aux = {'residuals': residuals, 'alpha': [st[c, 0].float() for c in range(C)],
               'reg_energy': [st[c, 3].float() for c in range(C)]}
        return loss_terms, out, aux

    # -- the loop around it (reference trainer.py:358-476) -------------------------------------------------------------
    def _run_MCMC(self, data_loss=None, reg_loss=None, speed_test_iters=100, with_ASD=False, with_R_hat=False,
                  with_seg_posterior=False, with_jacobian_posterior=False, with_HD=False, HD_percentile=95.0, with_TRE=False):
        """burn-in + sampling; returns {'mean','std_dev', 'im_mean','im_std', 'n', 'DSC', 'ASD', 'no_non_diffeomorphic_voxels',
        'samples_per_sec'}; posterior statistics are over the kept samples of ALL ranks.  'ASD' (average surface distance,
        reference utils/util.py:171-176 through SimpleITK on the host): with_ASD=True computes it per kept sample on the device
        (utils.util.calc_metrics -> calc_ASD_GPU: one host synchronisation per sample, parity with SimpleITK unpinned), a
        (chains, structures) array per kept sample; otherwise the entry is a string saying that it was not computed.

        with_R_hat=True adds 'R_hat', the convergence check of the chains (split R-hat, BDA3 section 11.4, over the N kept
        samples of every chain of every rank: M = 2 x chains sequences of floor(N/2) draws):
          'displacement' (3,D,H,W), 'im' (1,D,H,W)  voxel-wise R-hat maps (SGLDSampler.convergence_diagnostics)
          'mask'    per component over the fixed mask: max R-hat and the voxel counts above 1.01 and 1.1
          'traces'  {'data', 'reg', 'alpha', 'reg_energy'} -> {'R_hat', 'ESS'} of the per-chain scalars at the kept samples
                    (utils.diagnostics.split_rhat / ess), 'n' and 'M'
        With save_dir, MCMC_R_hat_displacement.vtk and MCMC_R_hat_im.nii.gz are written as well.  The per-chain accumulators
        take 64 C V bytes while the run lasts.  In hyper_mode='reference' (the default) the chains share the mixture and
        regulariser parameters that they step in turn, so they are not independent: R-hat is still computed, but its reading
        as a check between independent chains holds for hyper_mode 'per_chain' / 'frozen' (Trainer(sampler_config=...)).
        With with_R_hat=False nothing of this runs and the result is unchanged.

        with_seg_posterior=True (needs structures_dict and fixed and moving segmentations, else ValueError) adds
        'seg_posterior', the posterior of the warped moving segmentation over every kept sample of every chain of every rank
        (SGLDSampler.enable_segmentation_posterior over the structures' labels; the segmentation warped for the Dice scores is
        folded into the label counts): the maps 'probability' (L,D,H,W), 'majority' (1,1,D,H,W) int16, 'entropy' (1,D,H,W),
        'labels', 'n', 'summary' (L,3) int64, and 'structures' {name: {'expected_volume' (voxels), 'uncertain_voxels',
        'soft_DSC', 'DSC_majority'[, 'ASD_majority' with with_ASD]}}.  With save_dir, MCMC_seg_majority.nii.gz and
        MCMC_seg_entropy.nii.gz are written as well.  With with_seg_posterior=False nothing of this runs.

        with_jacobian_posterior=True adds 'jacobian_posterior', the posterior of log det J of the transformation over every kept
        sample of every chain of every rank (SGLDSampler.enable_jacobian_posterior; a sample is folded at a voxel where log det
        J is not finite): the maps 'fold_probability', 'log_det_J_mean', 'log_det_J_std' (D,H,W), 'n', and over the fixed mask
        'expected_folded_voxels' (sum of the folding probabilities), 'voxels_ever_folded', 'voxels_folded_in_majority',
        'mean_log_det_J', 'mean_std_log_det_J', plus per kept sample and chain (all ranks' chains) 'SDlogJ', the population std
        of log det J over the finite mask voxels, and 'folded_fraction', the folded share of the mask, as (kept samples,
        chains) arrays.  Registration challenges that report SDlogJ clip det J at 1e-9 instead of leaving the non-positive
        voxels out.  With save_dir, MCMC_log_det_J_mean.nii.gz, MCMC_log_det_J_std_dev.nii.gz and
        MCMC_fold_probability.nii.gz are written as well.  With with_jacobian_posterior=False nothing of this runs.

        with_HD=True adds 'HD' and 'HD95' (the key follows HD_percentile: 'HD99' for 99), one (chains, structures) array per
        kept sample like 'ASD': the Hausdorff distance of the label contours and the larger of the two directed percentiles
        of the contour distances (numpy's default percentile; utils.util.calc_HD_GPU, the label-contour / distance transform
        kernels of the ASD plus a radix select on the device).  With with_ASD as well, one distance transform per kept sample
        gives all three.  With with_seg_posterior, the structures also get 'HD_majority' and 'HD95_majority'.  With
        with_HD=False nothing of this runs.

        with_TRE=True (needs 'landmarks' in both the fixed and the moving dict: (P,3) zero-based (x, y, z) voxel coordinates,
        row i of one corresponding to row i of the other, else ValueError) adds 'TRE', the mean target registration error
        (mm, spacing im_spacing) of the landmarks per kept sample and chain of every rank, a (kept samples, chains) array, and
        'landmark_posterior' (SGLDSampler.enable_landmark_posterior, over every kept sample of every chain of every rank): the
        per-landmark arrays 'mean_position' (moving voxels), 'TRE_of_mean', 'expected_TRE', 'TRE_std', 'covariance' (P,6)
        mm^2, 'principal_std' (P,3) mm, 'mahalanobis2', the summaries 'mean_TRE_of_mean', 'mean_expected_TRE',
        'initial_TRE' / 'mean_initial_TRE' (the identity transformation), 'coverage' {50, 90, 95: share of the true moving
        landmarks inside the posterior's credible ellipsoid of that level}, 'uncertainty_error_spearman' (rank correlation of
        sqrt(trace covariance) with the TRE of the mean), and 'TRE_max' / 'TRE_std' (max and population std over the
        landmarks) per kept sample and chain.  With save_dir, MCMC_landmarks.vtk is written as well.  With with_TRE=False
        nothing of this runs."""
        if self.SGLD_params is None:
            self._SGLD_init()
        s = self.sampler
        if with_seg_posterior:
            if not (self.structures_dict and s.moving_seg is not None and 'seg' in self.fixed):
                raise ValueError('with_seg_posterior=True needs structures_dict and fixed and moving segmentations')
            s.enable_segmentation_posterior(list(self.structures_dict.values()))
        if with_jacobian_posterior:
            s.enable_jacobian_posterior()
        if with_TRE:
            s.enable_landmark_posterior(*self._landmark_pair(), self.im_spacing)
        if not self._gmm_pushed:
            if data_loss is not None or reg_loss is not None:
                self._push_hyper(data_loss, reg_loss)
                self._gmm_pushed = True
            else:
                self._GMM_init()
        dsc, asd, folded, hd, hd_q = [], [], [], [], []
        total = self.no_iters_burn_in + self.no_samples_MCMC
        if with_R_hat:
            n_kept = sum(1 for i in range(1, total + 1) if self._is_kept(i))
            s.enable_convergence_diagnostics(n_kept)
            # per kept sample, this rank's rows of the stats (alpha, data, reg, reg energy): a device copy, no synchronisation
            traces = torch.zeros(n_kept, self.no_chains, 4, device=s.device, dtype=torch.float64)
            k_kept = 0
        if with_jacobian_posterior:
            # per kept sample, this rank's rows of the Jacobian sums over the mask: a device copy, no synchronisation
            jac_traces = torch.zeros(sum(1 for i in range(1, total + 1) if self._is_kept(i)), self.no_chains, 4,
                                     device=s.device, dtype=torch.float64)
            k_jac = 0
        if with_TRE:
            # per kept sample, this rank's rows of the landmark TRE sums: a device copy, no synchronisation
            lm_traces = torch.zeros(sum(1 for i in range(1, total + 1) if self._is_kept(i)), self.no_chains, 3,
                                    device=s.device, dtype=torch.float64)
            k_lm = 0
        from ..utils.diff_op import GradientOperator
        diff_op = GradientOperator()
        it = 0
        while it < total:
            # run up to the next kept sample in one go (graph replays, no host involvement)
            nxt = it + 1
            while nxt <= total and not self._is_kept(nxt):
                nxt += 1
            nxt = min(nxt, total)
            s.step(nxt - it)
            it = nxt
            if self._is_kept(it):
                T = s.transformation()
                seg_w = None
                if self.structures_dict and s.moving_seg is not None and 'seg' in self.fixed:
                    seg_w = s.warp_segmentation(transformation=T)
                    seg_f = self.fixed['seg'].to(s.device).expand(self.no_chains, -1, -1, -1, -1)
                    dsc.append(calc_DSC_GPU(self.no_chains, seg_f, seg_w, self.structures_dict))
                    if with_ASD and not with_HD:
                        from ..utils.util import calc_metrics
                        asd.append(calc_metrics(seg_f, seg_w, self.structures_dict, self.im_spacing, no_samples=self.no_chains)[0])
                    elif with_HD:
                        ASD, HD, HD_q = self._surface_distances(seg_f, seg_w, self.no_chains, with_ASD, HD_percentile)
                        if with_ASD:
                            asd.append(ASD)
                        hd.append(HD)
                        hd_q.append(HD_q)
                # after the segmentation warp, so that the segmentation posterior reuses it; the transformation and the warp
                # read what accumulate() reads and write nothing it reads, so the order changes no result
                s.accumulate(seg_warped=seg_w, transformation=T)
                if with_R_hat:
                    traces[k_kept].copy_(s.stats[:, :4])
                    k_kept += 1
                if with_jacobian_posterior:
                    jac_traces[k_jac].copy_(s.last_jacobian_stats)
                    k_jac += 1
                if with_TRE:
                    lm_traces[k_lm].copy_(s.last_landmark_stats)
                    k_lm += 1
                n_folded, log_det_J = calc_no_non_diffeomorphic_voxels(T, diff_op)
                folded.append(n_folded)
                if self.save_dir is not None:
                    from ..logger import save_sample
                    for c in range(self.no_chains):
                        save_sample(self.save_dir, self.im_spacing, it, s.im_warped[c:c + 1], s.displacement[c:c + 1],
                                    log_det_J[c:c + 1], model='MCMC', chain_no=s.chain_offset + c)
                bad = bool((n_folded > 0.001 * self.no_voxels).any())
                if parallel.any_rank(bad, s.device):   # reference trainer.py:441-445 (exits the process there)
                    # the flag is all-reduced first: every rank leaves together instead of one raising while the others
                    # wait for it in the moments merge
                    raise RuntimeError(f'sample {it}: {n_folded} voxels where the sampled transformation is not '
                                       f'diffeomorphic' + ('' if bad else ' (on another rank)'))
        if data_loss is not None or reg_loss is not None:
            self._pull_hyper(data_loss, reg_loss)
        mom = s.posterior_moments()
        result = {'mean': mom['displacement_mean'], 'std_dev': mom['displacement_std'], 'im_mean': mom['im_mean'],
                  'im_std': mom['im_std'], 'n': mom['n'], 'DSC': dsc, 'no_non_diffeomorphic_voxels': folded,
                  'ASD': asd if with_ASD else 'unavailable: not requested (with_ASD=True computes the label-contour average '
                                              'Hausdorff distance of reference utils/util.py:171-176 per kept sample with the CUDA '
                                              'distance transform kernels; parity with SimpleITK unpinned)'}
        if with_HD:
            with_seg = bool(self.structures_dict and s.moving_seg is not None and 'seg' in self.fixed)
            result.update(self._HD_entries(hd, hd_q, with_seg, HD_percentile))
        if with_R_hat:
            result['R_hat'] = self._R_hat(traces)
        if with_seg_posterior:
            post = s.segmentation_posterior(seg_fixed=self.fixed['seg'])
            s.disable_segmentation_posterior()
            result['seg_posterior'] = self._seg_posterior(post, with_ASD, 'MCMC', with_HD, HD_percentile)
        if with_jacobian_posterior:
            post = s.jacobian_posterior()
            s.disable_jacobian_posterior()
            result['jacobian_posterior'] = self._jacobian_posterior(post, jac_traces, 'MCMC')
        if with_TRE:
            post = s.landmark_posterior()
            s.disable_landmark_posterior()
            result['TRE'], result['landmark_posterior'] = self._landmark_posterior(post, lm_traces, 'MCMC')
        if self.save_dir is not None and (not torch.distributed.is_initialized() or torch.distributed.get_rank() == 0):
            # MCMC_sample_{mean,std_dev}[_masked].vtk like the reference (trainer.py:457-460, logger/logger.py:110-131)
            from ..logger import save_displacement_mean_and_std_dev
            save_displacement_mean_and_std_dev(self.save_dir, self.im_spacing, mom['displacement_mean'], mom['displacement_std'],
                                               self.moving.get('mask'), 'MCMC')
        if speed_test_iters:  # the reference's built-in speed test: transitions + one segmentation warp each (:467-476)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(speed_test_iters):
                s.step(1)
                if s.moving_seg is not None:
                    s.warp_segmentation()
            torch.cuda.synchronize()
            result['samples_per_sec'] = self.no_chains * speed_test_iters / (time.perf_counter() - t0)
        return result

    @staticmethod
    def _HD_key(percentile):
        """'HD95' for the 95th percentile, 'HD99.5' for 99.5"""
        return f'HD{float(percentile):g}'

    def _surface_distances(self, seg_fixed, seg_warped, no_samples, with_ASD, percentile):
        """(ASD or None, HD, HD_q) of the warped segmentations, (no_samples, structures) each: one distance transform for all
        three when with_ASD (the ASD is calc_ASD_GPU's to the bit), calc_HD_GPU otherwise"""
        from ..utils.util import calc_HD_GPU, calc_surface_distances_GPU
        if with_ASD:
            return calc_surface_distances_GPU(no_samples, seg_fixed, seg_warped, self.structures_dict, self.im_spacing,
                                              percentile)
        return (None,) + calc_HD_GPU(no_samples, seg_fixed, seg_warped, self.structures_dict, self.im_spacing, percentile)

    def _HD_entries(self, hd, hd_q, available, percentile):
        """the 'HD' and 'HD95' entries of _run_MCMC / _test_VI(with_HD=True)"""
        if not available:
            why = 'unavailable: no segmentations / structures'
            return {'HD': why, self._HD_key(percentile): why}
        return {'HD': hd, self._HD_key(percentile): hd_q}

    def _R_hat(self, traces):
        """the 'R_hat' entry of _run_MCMC(with_R_hat=True) from the filled accumulators and this rank's traces (N, C, 4); frees
        the accumulators"""
        from .. import _lib as L
        from ..utils.diagnostics import ess, split_rhat
        s = self.sampler
        diag = s.convergence_diagnostics()
        s.disable_convergence_diagnostics()
        # all ranks' traces at their global chain offsets, gathered with one SUM all-reduce of a zero-padded buffer
        allt = torch.zeros(traces.shape[0], self.no_chains_total, 4, device=traces.device, dtype=torch.float64)
        allt[:, s.chain_offset:s.chain_offset + self.no_chains] = traces
        if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            torch.distributed.all_reduce(allt, op=torch.distributed.ReduceOp.SUM)
        allt = allt.cpu().numpy()
        cols = {'data': L.STAT_DATA, 'reg': L.STAT_REG, 'alpha': L.STAT_ALPHA, 'reg_energy': L.STAT_ENERGY}
        diag['traces'] = {name: {'R_hat': split_rhat(allt[:, :, j].T), 'ESS': ess(allt[:, :, j].T)} for name, j in cols.items()}
        if self.save_dir is not None and (not torch.distributed.is_initialized() or torch.distributed.get_rank() == 0):
            import os
            from ..logger import save_field_to_disk, save_im_to_disk
            os.makedirs(self.save_dir, exist_ok=True)
            sp = [float(x) for x in self.im_spacing]
            save_field_to_disk(diag['displacement'].cpu(), os.path.join(self.save_dir, 'MCMC_R_hat_displacement.vtk'), sp)
            save_im_to_disk(diag['im'][0].cpu(), os.path.join(self.save_dir, 'MCMC_R_hat_im.nii.gz'), sp)
        return diag

    def _seg_posterior(self, post, with_ASD, model, with_HD=False, HD_percentile=95.0):
        """the 'seg_posterior' entry of _run_MCMC / _test_VI(with_seg_posterior=True) from the dict of
        SGLDSampler.segmentation_posterior (computed with the fixed segmentation): per structure the expected volume S / n, the
        uncertain voxels U, the soft Dice 2 O / (S + n |F|) of the probability map and the Dice (and ASD, and with with_HD the
        Hausdorff distance and its percentile: 'HD_majority', 'HD95_majority') of the majority segmentation;
        {model}_seg_majority.nii.gz and {model}_seg_entropy.nii.gz in save_dir"""
        from .. import ops
        from ..utils.util import calc_ASD_GPU
        n, labels, majority = post['n'], post['labels'], post['majority']
        seg_f = self.fixed['seg'].to(majority.device).contiguous()
        summary = post['summary'].cpu().numpy()
        fixed_sizes = ops.dice_counts(seg_f, seg_f, labels)[0, :, 0].cpu().numpy()   # |F_l|
        dsc = calc_DSC_GPU(1, seg_f, majority, self.structures_dict)[0]
        if with_HD:   # one distance transform for the ASD and both Hausdorff figures
            asd, hd, hd_q = (None if x is None else x[0]
                             for x in self._surface_distances(seg_f, majority, 1, with_ASD, HD_percentile))
        else:
            asd = calc_ASD_GPU(1, seg_f, majority, self.structures_dict, self.im_spacing)[0] if with_ASD else None
        structures = {}
        for j, name in enumerate(self.structures_dict):
            S, O, U = (int(x) for x in summary[j])
            den = S + n * int(fixed_sizes[j])
            structures[name] = {'expected_volume': S / n, 'uncertain_voxels': U,
                                'soft_DSC': 2.0 * O / den if den else float('nan'), 'DSC_majority': float(dsc[j])}
            if with_ASD:
                structures[name]['ASD_majority'] = float(asd[j])
            if with_HD:
                structures[name]['HD_majority'] = float(hd[j])
                structures[name][f'{self._HD_key(HD_percentile)}_majority'] = float(hd_q[j])
        post['structures'] = structures
        if self.save_dir is not None and (not torch.distributed.is_initialized() or torch.distributed.get_rank() == 0):
            import os
            from ..logger import save_im_to_disk
            os.makedirs(self.save_dir, exist_ok=True)
            sp = [float(x) for x in self.im_spacing]
            save_im_to_disk(majority[0, 0].cpu(), os.path.join(self.save_dir, f'{model}_seg_majority.nii.gz'), sp)
            save_im_to_disk(post['entropy'][0].cpu(), os.path.join(self.save_dir, f'{model}_seg_entropy.nii.gz'), sp)
        return post

    def _jacobian_posterior(self, post, traces, model, gather=True):
        """the 'jacobian_posterior' entry of _run_MCMC / _test_VI(with_jacobian_posterior=True) from the dict of
        SGLDSampler.jacobian_posterior and this rank's per-sample rows (N, C, 4) = (finite, folded, sum ld, sum ld^2) over the
        mask; with gather, all ranks' rows at their global chain offsets (one SUM all-reduce of a zero-padded buffer, as the
        R-hat traces).  {model}_log_det_J_mean.nii.gz, {model}_log_det_J_std_dev.nii.gz and {model}_fold_probability.nii.gz
        in save_dir"""
        if gather:
            s = self.sampler
            allt = torch.zeros(traces.shape[0], self.no_chains_total, 4, device=traces.device, dtype=torch.float64)
            allt[:, s.chain_offset:s.chain_offset + self.no_chains] = traces
            if torch.distributed.is_available() and torch.distributed.is_initialized() and \
                    torch.distributed.get_world_size() > 1:
                torch.distributed.all_reduce(allt, op=torch.distributed.ReduceOp.SUM)
            traces = allt
        t = traces.cpu().numpy()
        finite, fold, s1, s2 = t[..., 0], t[..., 1], t[..., 2], t[..., 3]
        with np.errstate(divide='ignore', invalid='ignore'):
            m = s1 / finite
            post['SDlogJ'] = np.sqrt(np.maximum(s2 / finite - m * m, 0.0))   # population std; NaN without a finite voxel
            post['folded_fraction'] = fold / (finite + fold)
        summ = post['summary']
        post['expected_folded_voxels'] = summ['sum_folds'] / post['n']
        for key in ('voxels_ever_folded', 'voxels_folded_in_majority', 'mean_log_det_J', 'mean_std_log_det_J'):
            post[key] = summ[key]
        if self.save_dir is not None and (not torch.distributed.is_initialized() or torch.distributed.get_rank() == 0):
            import os
            from ..logger import save_im_to_disk
            os.makedirs(self.save_dir, exist_ok=True)
            sp = [float(x) for x in self.im_spacing]
            for key, name in (('log_det_J_mean', 'log_det_J_mean'), ('log_det_J_std', 'log_det_J_std_dev'),
                              ('fold_probability', 'fold_probability')):
                save_im_to_disk(post[key].cpu(), os.path.join(self.save_dir, f'{model}_{name}.nii.gz'), sp)
        return post

    def _landmark_pair(self):
        """the (fixed, moving) landmark tables of the image dicts, (P,3) each"""
        p, q = self.fixed.get('landmarks'), self.moving.get('landmarks')
        if p is None or q is None:
            raise ValueError("with_TRE=True needs 'landmarks' in both the fixed and the moving dict")
        if tuple(p.shape) != tuple(q.shape) or p.dim() != 2 or p.shape[1] != 3:
            raise ValueError(f'fixed and moving landmarks must both be (P, 3) with the same P: {tuple(p.shape)} vs '
                             f'{tuple(q.shape)}')
        return p, q

    def _landmark_posterior(self, post, traces, model, gather=True):
        """('TRE', 'landmark_posterior') of _run_MCMC / _test_VI(with_TRE=True) from the dict of
        SGLDSampler.landmark_posterior and this rank's per-sample rows (N, C, 3) = (sum TRE, sum TRE^2, max TRE); with gather,
        all ranks' rows at their global chain offsets (one SUM all-reduce of a zero-padded buffer, as the R-hat traces).
        {model}_landmarks.vtk in save_dir: the mean positions in mm, the covariance, E[TRE], the TRE of the mean and d^2"""
        from ..utils.util import landmark_posterior_summary
        if gather:
            s = self.sampler
            allt = torch.zeros(traces.shape[0], self.no_chains_total, 3, device=traces.device, dtype=torch.float64)
            allt[:, s.chain_offset:s.chain_offset + self.no_chains] = traces
            if torch.distributed.is_available() and torch.distributed.is_initialized() and \
                    torch.distributed.get_world_size() > 1:
                torch.distributed.all_reduce(allt, op=torch.distributed.ReduceOp.SUM)
            traces = allt
        t = traces.cpu().numpy()
        P = post['table'].shape[0]
        mean = t[..., 0] / P
        out = landmark_posterior_summary(post['table'], post['fixed_landmarks'], post['moving_landmarks'], post['spacing'])
        out['n'] = post['n']
        out['TRE_max'] = t[..., 2]
        out['TRE_std'] = np.sqrt(np.maximum(t[..., 1] / P - mean * mean, 0.0))   # population std over the landmarks
        if self.save_dir is not None and (not torch.distributed.is_initialized() or torch.distributed.get_rank() == 0):
            import os
            from ..logger import save_landmarks_to_disk
            os.makedirs(self.save_dir, exist_ok=True)
            sp = np.asarray(post['spacing'], dtype=np.float64)
            save_landmarks_to_disk(os.path.join(self.save_dir, f'{model}_landmarks.vtk'), out['mean_position'] * sp,
                                   out['covariance'], {'expected_TRE': out['expected_TRE'], 'TRE_of_mean': out['TRE_of_mean'],
                                                       'mahalanobis2': out['mahalanobis2']})
        return mean, out

    def _is_kept(self, sample_no):
        """reference trainer.py:414-415"""
        return sample_no > self.no_iters_burn_in and (sample_no % self.log_period_MCMC == 0 or
                                                      sample_no == self.no_samples_MCMC)
