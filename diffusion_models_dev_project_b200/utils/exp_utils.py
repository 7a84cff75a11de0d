"""Factories with the reference's signatures (src/utils/exp_utils.py:99-332).

``get_standard_ray_trafo(config)`` returns the CUDA-kernel operator for
``trafo_name='simple_trafo'`` whatever ``forward_op.impl`` says (there is one
implementation); the optional keys ``forward_op.angle_range`` (a limited-angle wedge)
and ``forward_op.angles`` (an explicit, possibly non-uniform view set) select other
angle sets.  ``get_standard_sampler`` keeps the reference's signature but
builds the DDPM/'dds' sampler correctly: the reference passes an
``init_chain_fn`` keyword ``BaseSampler`` does not accept and therefore raises
(exp_utils.py:214-221, see SURVEY.md §3.1); only the branch the hot path needs
-- ``method='dds'`` -- is provided, other methods raise ``NotImplementedError``.
"""
import functools
from math import ceil

import torch

from .sde import VESDE, VPSDE, DDPM, _EPSILON_PRED_CLASSES
from ..physics import B200RayTrafo, simulate
from ..physics.geometry import ParallelBeamGeometry2D
from ..samplers import (BaseSampler, decomposed_diffusion_sampling_sde_predictor,
                        adapted_ddim_sde_predictor, tv_loss, adaptation_loss, AdaptationLoss, _adapt, _score_model_adpt,
                        Euler_Maruyama_sde_predictor, Ancestral_Sampling)


def get_standard_sde(config):
    name = config.sde.type.lower()
    if name == 'vesde':
        return VESDE(sigma_min=config.sde.sigma_min, sigma_max=config.sde.sigma_max)
    if name == 'vpsde':
        return VPSDE(beta_min=config.sde.beta_min, beta_max=config.sde.beta_max)
    if name == 'ddpm':
        return DDPM(beta_min=config.sde.beta_min, beta_max=config.sde.beta_max, num_steps=config.sde.num_steps)
    raise NotImplementedError(name)


def _optional(ns, key):
    """``ns.key`` or None: config objects signal a missing key with AttributeError (namespaces, ConfigDict) or
    KeyError (dicts with attribute access)."""
    try:
        return getattr(ns, key)
    except (AttributeError, KeyError):
        return None


def get_standard_ray_trafo(config):
    """``forward_op.angle_range = (min, max)`` (radians): ``num_angles`` cell-centred views on ``[min, max)``.
    ``forward_op.angles`` (radians): exactly these views, weighted by their angular cells (``num_angles`` may be
    omitted; if given it must equal their count).  Without either key: ``num_angles`` views on ``[0, pi)``."""
    fo = config.forward_op
    if fo.trafo_name.lower() != 'simple_trafo':
        raise NotImplementedError(fo.trafo_name)
    im_shape = (config.data.im_size, config.data.im_size)
    angle_range = _optional(fo, 'angle_range')
    angles = _optional(fo, 'angles')
    if angle_range is not None and angles is not None:
        raise ValueError('forward_op: give angle_range or angles, not both')
    if angles is not None:
        geom = ParallelBeamGeometry2D.from_angles(im_shape, angles)
        num_angles = _optional(fo, 'num_angles')
        if num_angles is not None and int(num_angles) != geom.n_angles:
            raise ValueError('forward_op.num_angles = %d but %d angles are given' % (int(num_angles), geom.n_angles))
        return B200RayTrafo(im_shape=im_shape, num_angles=geom.n_angles, impl=fo.impl, geometry=geom)
    if angle_range is not None:
        return B200RayTrafo(im_shape=im_shape, num_angles=fo.num_angles, impl=fo.impl,
                            angle_range=tuple(float(a) for a in angle_range))
    return B200RayTrafo(im_shape=im_shape, num_angles=fo.num_angles, impl=fo.impl)


def get_data_from_ground_truth(ground_truth, ray_trafo, white_noise_rel_stddev):
    ground_truth = ground_truth.unsqueeze(0) if ground_truth.ndim == 3 else ground_truth
    observation = simulate(x=ground_truth, ray_trafo=ray_trafo,
                           white_noise_rel_stddev=white_noise_rel_stddev, return_noise_level=False)
    filtbackproj = ray_trafo.fbp(observation)
    return ground_truth, observation, filtbackproj


def _im_shape_of(ray_trafo):
    return ray_trafo.im_shape if not hasattr(ray_trafo, 'resize') else ray_trafo.resize.shape


def get_standard_sampler(args, config, score, sde, ray_trafo, observation=None, filtbackproj=None, device=None):
    """Sampler factory with the reference's signature (src/utils/exp_utils.py:123-223).

    ``dds`` (the data-consistency hot path) for every schedule; ``dps`` = diffusion posterior
    sampling (Euler-Maruyama for VE/VP, ancestral for DDPM); ``naive`` = score + data-fit gradient
    (VE/VP only, as in the reference).  The reference passes an undefined ``init_chain_fn`` on the
    VE/VP branch; here the chain always starts from the prior."""
    method = args.method.lower()
    shape = _im_shape_of(ray_trafo)
    eps_pred = any(isinstance(sde, c) for c in _EPSILON_PRED_CLASSES)
    sample_kwargs = {
        'num_steps': int(args.num_steps),
        'batch_size': config.sampling.batch_size,
        'start_time_step': ceil(float(args.pct_chain_elapsed) * int(args.num_steps)),
        'im_shape': [config.model.in_channels, *shape],
        'eps': config.sampling.eps,
    }

    def nloglik(x):
        return torch.linalg.norm(observation - ray_trafo(x))

    if method == 'dds':
        sample_kwargs['predictor'] = {'eta': float(args.eta), 'gamma': float(args.gamma),
                                      'use_simplified_eqn': True, 'ray_trafo': ray_trafo}
        predictor = functools.partial(
            decomposed_diffusion_sampling_sde_predictor, score=score, sde=sde,
            rhs=ray_trafo.trafo_adjoint(observation), cg_kwargs={'max_iter': int(args.cg_iter)})
    elif method == 'dps' and eps_pred:
        sample_kwargs['predictor'] = {'penalty': float(args.penalty)}
        sample_kwargs['early_stopping_pct'] = float(args.early_stopping_pct)
        predictor = functools.partial(Ancestral_Sampling, nloglik=nloglik)
    elif method in ('dps', 'naive') and not eps_pred:
        sample_kwargs['predictor'] = {'aTweedy': method == 'dps', 'penalty': float(args.penalty)}
        predictor = functools.partial(Euler_Maruyama_sde_predictor, nloglik=nloglik)
    else:
        raise NotImplementedError(method)
    if eps_pred:
        sample_kwargs['travel_length'] = config.sampling.travel_length
        sample_kwargs['travel_repeat'] = config.sampling.travel_repeat
        assert sample_kwargs['start_time_step'] == 0
    return BaseSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=sample_kwargs,
                       device=device if device is not None else config.device)


def get_standard_adapted_sampler(args, config, score, sde, ray_trafo, observation=None, device=None,
                                 complex_y=False, lora_inject_fn=None):
    if args.method.lower() != 'dds':
        raise NotImplementedError
    eps = getattr(config.sampling, 'eps', 0.)
    shape = _im_shape_of(ray_trafo)
    sample_kwargs = {
        'num_steps': int(args.num_steps),
        'batch_size': config.sampling.batch_size,
        'start_time_step': 0,
        'im_shape': [config.model.in_channels, *shape],
        'eps': eps,
        'adapt_freq': int(args.adapt_freq),
        'predictor': {'eta': float(args.eta), 'use_simplified_eqn': True, 'gamma': float(args.gamma),
                      'ray_trafo': ray_trafo},
        'corrector': {},
        'early_stopping_pct': float(args.early_stopping_pct),
    }
    adpt_kwargs = None
    if args.adaptation == 'lora':
        adpt_kwargs = {'include_blocks': args.lora_include_blocks, 'r': int(args.lora_rank)}
    _score_model_adpt(score, impl=args.adaptation, adpt_kwargs=adpt_kwargs, inject_fn=lora_inject_fn)

    loss_fn = AdaptationLoss(observation, ray_trafo, float(args.tv_penalty))     # callable: loss_fn(x=...)

    adapt_fn = functools.partial(_adapt, score=score, sde=sde, loss_fn=loss_fn,
                                 num_steps=int(args.num_optim_step), lr=float(args.lr),
                                 cuda_graph=getattr(args, 'adapt_cuda_graph', None))
    predictor = functools.partial(
        adapted_ddim_sde_predictor, score=score, sde=sde, adapt_fn=adapt_fn, add_cg=args.add_cg,
        dc_type=args.dc_type, rhs=ray_trafo.trafo_adjoint(observation),
        cg_kwargs={'max_iter': int(args.cg_iter)})
    if any(isinstance(sde, c) for c in _EPSILON_PRED_CLASSES):
        try:
            tl, tr = config.sampling.travel_length, config.sampling.travel_repeat
        except AttributeError:
            tl, tr = config.time_travel.travel_length, config.time_travel.travel_repeat
        sample_kwargs.update({'travel_length': tl, 'travel_repeat': tr})
    return BaseSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=sample_kwargs,
                       device=device if device is not None else config.device)
