"""
ctypes binding of libirsgmcmc.so (C ABI declared in include/irsgmcmc.h).

There is no fallback: if the shared library is missing or a CUDA device is not available, every op raises.  PyTorch is
used for device memory and streams only -- pointers are passed as integers, launches go to torch's current stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# IRSGMCMC_LIB: development override (A/B builds of the same library; irsgmcmc_b200/build.py `out=`)
LIB_PATH = os.environ.get('IRSGMCMC_LIB') or os.path.join(_HERE, 'libirsgmcmc.so')

c_float_p = ctypes.c_void_p
HYPER_SIZE = 96
STAT_SIZE = 8
MAX_K = 8

# offsets into the `hyper` array (include/irsgmcmc.h)
HYPER_GMM_STEP, HYPER_LOG_STD, HYPER_LOGITS = 0, 1, 9
HYPER_M_LOG_STD, HYPER_V_LOG_STD, HYPER_M_LOGITS, HYPER_V_LOGITS = 17, 25, 33, 41
HYPER_REG_STEP, HYPER_REG_P, HYPER_REG_M, HYPER_REG_V, HYPER_ITER = 49, 50, 52, 54, 56
HYPER_GMM_BETA_POW, HYPER_REG_BETA_POW = 57, 59
STAT_ALPHA, STAT_DATA, STAT_REG, STAT_ENERGY, STAT_NLL_PRE, STAT_REG_COEF = 0, 1, 2, 3, 4, 5

DATA_LCC, DATA_SSD = 0, 1
HYPER_MODES = {'reference': 0, 'per_chain': 1, 'frozen': 2}
REG_L2, REG_LOGNORMAL = 0, 1


class SgldConfig(ctypes.Structure):
    _fields_ = [('C', ctypes.c_int), ('D', ctypes.c_int), ('H', ctypes.c_int), ('W', ctypes.c_int),
                ('chain_offset', ctypes.c_int), ('data_term', ctypes.c_int), ('K', ctypes.c_int),
                ('lcc_s', ctypes.c_int), ('reg_type', ctypes.c_int), ('reg_learnable', ctypes.c_int),
                ('n_taps', ctypes.c_int), ('svf_steps', ctypes.c_int), ('virtual_decimation', ctypes.c_int),
                ('use_jitter', ctypes.c_int), ('gather_radius_max', ctypes.c_int), ('hyper_mode', ctypes.c_int),
                ('taps', ctypes.c_float * 16),
                ('tau', ctypes.c_double), ('jitter_alpha', ctypes.c_double), ('w_reg', ctypes.c_double),
                ('dof', ctypes.c_double),
                ('lr_log_std', ctypes.c_double), ('lr_logits', ctypes.c_double), ('lr_reg0', ctypes.c_double),
                ('lr_reg1', ctypes.c_double), ('lr_decay', ctypes.c_double), ('beta1', ctypes.c_double),
                ('beta2', ctypes.c_double), ('adam_eps', ctypes.c_double),
                ('gmm_scale_prior_loc', ctypes.c_double), ('gmm_scale_prior_scale', ctypes.c_double),
                ('dirichlet_alpha', ctypes.c_double),
                ('reg_scale_prior_loc', ctypes.c_double), ('reg_scale_prior_scale', ctypes.c_double),
                ('w_reg_prior_shape', ctypes.c_double), ('w_reg_prior_rate', ctypes.c_double),
                ('n_mask', ctypes.c_double), ('seed', ctypes.c_ulonglong),
                ('ffd_cps', ctypes.c_int * 3), ('ffd_grid', ctypes.c_int * 3), ('ffd_kernel', (ctypes.c_float * 32) * 3)]


class SgldBuffers(ctypes.Structure):
    _fields_ = [('v', ctypes.c_void_p), ('sigma', ctypes.c_void_p), ('sigma_chain_stride', ctypes.c_longlong),
                ('fixed', ctypes.c_void_p), ('moving', ctypes.c_void_p), ('mask', ctypes.c_void_p),
                ('eps', ctypes.c_void_p), ('jitter_unit', ctypes.c_void_p),
                ('css', ctypes.c_void_p), ('hist', ctypes.c_void_p), ('im_warped', ctypes.c_void_p),
                ('z', ctypes.c_void_p), ('lcc_a', ctypes.c_void_p), ('lcc_rs', ctypes.c_void_p),
                ('scratch1', ctypes.c_void_p), ('scratch2', ctypes.c_void_p),
                ('field_a', ctypes.c_void_p), ('field_b', ctypes.c_void_p), ('grad_v', ctypes.c_void_p),
                ('maxabs', ctypes.c_void_p), ('hyper', ctypes.c_void_p), ('stats', ctypes.c_void_p),
                ('gmm_table', ctypes.c_void_p), ('partials', ctypes.c_void_p), ('counters', ctypes.c_void_p),
                ('ffd_dense', ctypes.c_void_p), ('ffd_grad', ctypes.c_void_p), ('ffd_scratch', ctypes.c_void_p),
                ('ffd_work', ctypes.c_void_p)]


class ViBuffers(ctypes.Structure):
    _fields_ = [('mu', ctypes.c_void_p), ('log_var', ctypes.c_void_p), ('u', ctypes.c_void_p),
                ('adam_m', ctypes.c_void_p * 3), ('adam_v', ctypes.c_void_p * 3), ('eps_store', ctypes.c_void_p),
                ('vi_state', ctypes.c_void_p), ('partials', ctypes.c_void_p), ('counter', ctypes.c_void_p),
                ('eps', ctypes.c_void_p), ('x', ctypes.c_void_p),
                ('lr_mu', ctypes.c_double), ('lr_log_var', ctypes.c_double), ('lr_u', ctypes.c_double),
                ('lr_decay', ctypes.c_double), ('beta1', ctypes.c_double), ('beta2', ctypes.c_double),
                ('adam_eps', ctypes.c_double)]


# average surface distance scratch (include/irsgmcmc.h): IRS_ASD_MAX_BOXES counters, IRS_ASD_PARTIALS_DOUBLES partials
ASD_MAX_BOXES, ASD_PARTIALS_DOUBLES = 48, 48 * 4 * 64
# Hausdorff distance (include/irsgmcmc.h): IRS_SD_COUNTERS counters (the ASD tickets and the two list lengths per box)
SD_COUNTERS = 3 * ASD_MAX_BOXES

# split R-hat (include/irsgmcmc.h): components per launch, reduction scratch
RHAT_MAX_COMPONENTS, RHAT_PARTIALS_DOUBLES = 4, 4 * 3 * 256

# Jacobian posterior (include/irsgmcmc.h): reduction scratch per chain, words of the finish's summary
JACOBIAN_REDUCE_BLOCKS, JACOBIAN_SUMMARY_WORDS = 1184, 8

# landmark posterior (include/irsgmcmc.h): accumulator doubles and posterior columns per landmark
LANDMARK_ACC, LANDMARK_COLS = 11, 16

VI_STATE_SIZE, VI_STEP, VI_BETA_POW, VI_X, VI_SUMS, VI_ENTROPY = 16, 0, 1, 3, 4, 8

# name -> (restype, argtypes); every symbol include/irsgmcmc.h declares
_vp, _i, _ll, _f, _d, _ull, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_double,
                                   ctypes.c_ulonglong, ctypes.c_size_t)
SYMBOLS = {
    'irs_abi_version': (_i, []),
    'irs_error_string': (ctypes.c_char_p, [_i]),
    'irs_warp3d_fwd': (_i, [_vp, _ll, _vp, _vp, _f, _vp, _i, _i, _i, _i, _vp]),
    'irs_warp3d_bwd_grid': (_i, [_vp, _ll, _vp, _vp, _f, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_warp3d_nearest_i16': (_i, [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_warp3d_nearest_u8': (_i, [_vp, _ll, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_svf_hist_floats': (_sz, [_i, _i, _i, _i, _i]),
    'irs_svf_maxabs_floats': (_sz, [_i, _i, _i, _i, _i]),
    'irs_svf_exp_fwd': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'irs_svf_outputs': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_svf_exp_bwd': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    'irs_ffd_work_floats': (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    'irs_ffd_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'irs_ffd_bwd': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'irs_bspline_axis': (_i, [_vp, _vp, _i, _ll, _i, _i, _ll, _vp, _i, _i, _vp]),
    'irs_langevin_sobolev': (_i, [_vp, _vp, _ll, _f, _vp, _ull, _ull, _i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_diff_fwd': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'irs_diff_bwd': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'irs_reduce_scratch_doubles': (_sz, [_i, _i, _i, _i]),
    'irs_reg_energy': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_reg_energy_grad': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_lcc_normalise': (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_lcc_normalise_bwd': (_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_gmm_log_pdf': (_i, [_vp, _ll, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'irs_vd_factor': (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'irs_vd_factor_residual': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'irs_log_det_jacobian': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'irs_dice_counts': (_i, [_vp, _ll, _vp, _vp, _i, _vp, _i, _ll, _vp]),
    'irs_surface_boxes': (_i, [_vp, _ll, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    'irs_average_surface_distance': (_i, [_vp, _ll, _vp, _vp, _i, _vp, _vp, _i, _i, _vp, _ll, _vp, _vp, _vp, _i, _i, _i, _i,
                                          _vp]),
    'irs_surface_distances': (_i, [_vp, _ll, _vp, _vp, _i, _vp, _vp, _d, _i, _i, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _i, _i, _i,
                                   _i, _vp]),
    'irs_welford_update': (_i, [_vp, _i, _ll, _d, _vp, _vp, _vp]),
    'irs_welford_std': (_i, [_vp, _d, _vp, _ll, _vp]),
    'irs_split_welford_update': (_i, [_vp, _vp, _i, _ll, _i, _d, _vp, _vp, _vp]),
    'irs_split_rhat_sums': (_i, [_vp, _vp, _i, _ll, _i, _vp, _vp]),
    'irs_split_rhat_between': (_i, [_vp, _i, _ll, _vp, _i, _vp, _vp]),
    'irs_split_rhat_finish': (_i, [_vp, _vp, _i, _i, _vp, _i, _ll, _vp, _vp, _vp, _vp, _vp]),
    'irs_label_counts_update': (_i, [_vp, _i, _ll, _vp, _i, _vp, _vp]),
    'irs_label_posterior': (_i, [_vp, _vp, _i, _ll, _ll, _vp, _vp, _vp, _vp, _vp, _vp]),
    'irs_jacobian_update': (_i, [_vp, _vp, _i, _i, _i, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'irs_jacobian_posterior': (_i, [_vp, _vp, _vp, _ll, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'irs_landmark_map': (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    'irs_landmark_update': (_i, [_vp, _vp, _i, _i, _d, _vp, _vp, _vp]),
    'irs_landmark_posterior': (_i, [_vp, _vp, _i, _ll, _vp, _vp, _vp]),
    'irs_sgld_partials_doubles': (_sz, [ctypes.POINTER(SgldConfig)]),
    'irs_sgld_step': (_i, [ctypes.POINTER(SgldConfig), ctypes.POINTER(SgldBuffers), _vp]),
    'irs_sgld_step_profile': (_i, [ctypes.POINTER(SgldConfig), ctypes.POINTER(SgldBuffers), _vp, _vp]),
    'irs_sgld_launches_per_step': (_i, [ctypes.POINTER(SgldConfig)]),
    'irs_sgld_gmm_init': (_i, [ctypes.POINTER(SgldConfig), ctypes.POINTER(SgldBuffers), _vp, _i, _vp]),
    'irs_masked_mean_std': (_i, [_vp, _vp, _ll, _vp, _vp, _vp, _vp]),
    'irs_vi_step': (_i, [ctypes.POINTER(SgldConfig), ctypes.POINTER(SgldBuffers), ctypes.POINTER(ViBuffers), _vp]),
}

_lib = None


def load():
    """load libirsgmcmc.so; raises (never falls back) when it has not been built"""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                           f'(irsgmcmc_b200 has no CPU or PyTorch fallback)')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    if lib.irs_abi_version() != 4:
        raise RuntimeError('libirsgmcmc.so ABI version mismatch')
    _lib = lib
    return lib


def check(code):
    if code != 0:
        raise RuntimeError(f'libirsgmcmc: {load().irs_error_string(code).decode()} (code {code})')


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    """the boundary checks of SURVEY section 8b: CUDA device, contiguous"""
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError('irsgmcmc_b200 ops need CUDA tensors: there is no CPU implementation')
        if not t.is_contiguous():
            raise RuntimeError('irsgmcmc_b200 ops need contiguous tensors')


def ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def host_floats(values):
    arr = (ctypes.c_float * len(values))(*[float(x) for x in values])
    return arr
