"""B200-native data-consistency hot path of the SCD / DDS reverse sampler.

Public surface (names follow the reference's ``src`` package):

    B200RayTrafo / SimpleTrafo, BaseRayTrafo, simulate, SimulatedDataset  (physics)
    cg, DDPM, VESDE, VPSDE, PSNR, SSIM                                  (utils)
    BaseSampler, decomposed_diffusion_sampling_sde_predictor,
    adapted_ddim_sde_predictor, _adapt, ddim, apTweedy, ...       (samplers)
    get_standard_{sde,ray_trafo,sampler,adapted_sampler}          (utils.exp_utils)
"""
from .physics import (BaseRayTrafo, B200RayTrafo, SimpleTrafo, NormalOp, MeasurementWeights, ParallelBeamGeometry2D, simulate,
                      simulate_poisson, SimulatedDataset)
from .utils import SDE, VESDE, VPSDE, DDPM, PSNR, SSIM, cg, _EPSILON_PRED_CLASSES, _SCORE_PRED_CLASSES
from .samplers import (BaseSampler, tv_loss, adaptation_loss, _score_model_adpt, apTweedy, ddim,
                       decomposed_diffusion_sampling_sde_predictor, adapted_ddim_sde_predictor,
                       _adapt, _schedule_jump, wrapper_ddim, Euler_Maruyama_sde_predictor, Ancestral_Sampling,
                       Langevin_sde_corrector)
from .utils.exp_utils import (get_standard_sde, get_standard_ray_trafo, get_standard_sampler,
                              get_standard_adapted_sampler, get_data_from_ground_truth,
                              get_low_dose_data_from_ground_truth)

__version__ = '0.1.0'
