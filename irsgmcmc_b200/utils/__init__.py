from .diff_op import DifferentialOperator, GradientOperator
from .functions import SGLD, SobolevGrad, Sobolev_kernel_1D, langevin_sobolev
from .registration import RegistrationModule
from .sampler import sample_q_v
from .transformation import (B_spline_1D_kernel, Cubic_B_spline_FFD_3D, SVF_3D, SVFFD_3D, TransformationModule, conv1D,
                             cubic_B_spline_1D_value)
from .util import (add_noise_Langevin, add_noise_uniform_field, calc_ASD_GPU, calc_ASD_host, calc_det_J, calc_DSC_GPU,
                   calc_HD_GPU, calc_HD_host, calc_metrics, calc_TRE_GPU, calc_TRE_host,
                   landmark_posterior_summary, calc_no_non_diffeomorphic_voxels,
                   calc_norm, calc_posterior_statistics, calc_VD_factor, get_control_grid_size, get_noise_Langevin, get_noise_uniform,
                   init_identity_grid_3D, rescale_residuals, separable_conv_3D, transform_coordinates,
                   transform_coordinates_inv)
