"""Adaptation helpers of SCD (reference src/samplers/adaptation.py)."""
from typing import Dict, Optional

import torch
from torch import nn


def tv_loss(x):
    """Anisotropic total variation on the cropped differences (reference :7-11)."""
    dh = torch.abs(x[..., :, 1:] - x[..., :, :-1])
    dw = torch.abs(x[..., 1:, :] - x[..., :-1, :])
    return torch.sum(dh[..., :-1, :] + dw[..., :, :-1])


class _AdaptationLossFn(torch.autograd.Function):
    """``mean((A x - y)^2) + lam * tv_loss(x)`` with hand-written forward and backward:
    A and the residual/TV reductions forward (5 launches), ``d tv/dx`` and one backprojection
    with the TV gradient as fused addend backward (3 launches).  The gradient through A follows the
    ODL ``OperatorFunction`` pairing used everywhere else: ``(2/N) * A*(r) / c_w`` (SURVEY.md 8b).
    With measurement weights ``wts`` the data term is ``mean(W (A x - y)^2)`` and ``r = W (A x - y)``."""

    @staticmethod
    def forward(ctx, x, y, rt, lam, wts=None):
        import ctypes as C
        from .. import _lib
        lib = _lib.load()
        x = rt._prep(x, rt.im_shape, 'adaptation loss')
        dev = x.device
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        ax = rt._fp(x)
        y = y.to(device=dev, dtype=torch.float32).expand_as(ax).contiguous()
        numel = ax.numel()
        r = torch.empty_like(ax)
        part = torch.empty(int(lib.scd_residual_sq_blocks(numel)), dtype=torch.float32, device=dev)
        images = x.numel() // (rt.im_shape[0] * rt.im_shape[1])
        tvp = torch.empty(images * int(lib.scd_tv_blocks(*rt.im_shape)), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            if wts is None:
                _lib.check(lib.scd_residual_sq(ax.data_ptr(), y.data_ptr(), r.data_ptr(), part.data_ptr(), numel, stream),
                           'scd_residual_sq')
            else:
                w = wts.expanded(x.shape[:-2])
                _lib.check(lib.scd_residual_sq_w(ax.data_ptr(), y.data_ptr(), w.data_ptr(), r.data_ptr(), part.data_ptr(),
                                                 numel, stream), 'scd_residual_sq_w')
            _lib.check(lib.scd_tv_loss(x.data_ptr(), tvp.data_ptr(), images, rt.im_shape[0], rt.im_shape[1], stream),
                       'scd_tv_loss')
        ctx.save_for_backward(x, r)
        ctx.rt, ctx.lam, ctx.numel, ctx.images = rt, float(lam), numel, images
        return part.sum() / numel + float(lam) * tvp.sum()

    @staticmethod
    def backward(ctx, g):
        import ctypes as C
        from .. import _lib
        lib = _lib.load()
        x, r = ctx.saved_tensors
        rt = ctx.rt
        dev = x.device
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        tvg = torch.empty_like(x)
        with torch.cuda.device(dev):
            _lib.check(lib.scd_tv_grad(x.data_ptr(), tvg.data_ptr(), ctx.images, rt.im_shape[0], rt.im_shape[1], stream),
                       'scd_tv_grad')
        # the gradient of the residual is the plain transpose of A: adj_scale/c_w = dx^2/ds times the unweighted
        # backprojection sum, so the view weights that scd_bp applies for A* are divided out first
        scale = 2.0 / ctx.numel * rt.adj_scale / rt.geometry.range_weight
        w = rt._view_weights(dev)
        grad = rt._bp(r if w is None else r / w, scale, addend=tvg, addend_scale=ctx.lam)
        return grad * g, None, None, None, None


def adaptation_loss(x, observation, ray_trafo, tv_penalty: float, weights=None):
    """The SCD adaptation loss (reference src/utils/exp_utils.py:256-257).  With a
    :class:`B200RayTrafo` and CUDA tensors it runs as fused kernels with a hand-written
    backward; any other ray transform evaluates the reference's tensor expression.
    ``weights`` (a :class:`MeasurementWeights` or a tensor): ``mean(W (A x - y)^2) + tv_penalty * tv(x)``."""
    from ..physics.b200_ray_trafo import B200RayTrafo, MeasurementWeights, as_weights
    if isinstance(ray_trafo, B200RayTrafo) and x.is_cuda and x.dtype == torch.float32:
        return _AdaptationLossFn.apply(x, observation, ray_trafo, float(tv_penalty), as_weights(ray_trafo, weights))
    res2 = (ray_trafo(x) - observation).pow(2)
    if weights is not None:
        res2 = (weights.w if isinstance(weights, MeasurementWeights) else weights) * res2
    return torch.mean(res2) + float(tv_penalty) * tv_loss(x)


class AdaptationLoss:
    """The loss closure of ``get_standard_adapted_sampler`` (reference src/utils/exp_utils.py:256-257) as an
    object, so that :func:`..samplers.utils._adapt` can recognise it and evaluate Tweedie -> data consistency ->
    loss and the whole backward sweep as two library calls (``scd_adapt_fwd`` / ``scd_adapt_bwd``).  Calling it
    evaluates the loss at ``x`` like the reference's lambda.  ``weights``: measurement weights ``W`` of the data
    term, ``mean(W (A x - y)^2)`` (:class:`MeasurementWeights` or a tensor for one); the data-consistency step of
    the adaptation objective then solves ``(I + gamma A*WA)`` as well."""

    def __init__(self, observation, ray_trafo, tv_penalty: float, weights=None):
        from ..physics.b200_ray_trafo import B200RayTrafo, as_weights
        self.observation, self.ray_trafo, self.tv_penalty = observation, ray_trafo, float(tv_penalty)
        self.weights = as_weights(ray_trafo, weights) if isinstance(ray_trafo, B200RayTrafo) else weights

    def __call__(self, x):
        return adaptation_loss(x, self.observation, self.ray_trafo, self.tv_penalty, self.weights)


_DC_CODES = {'cg': 0, 'dc': 1, 'gd': 1, 'none': 2}


class _AdaptObjectiveFn(torch.autograd.Function):
    """``loss(s) = AdaptationLoss(dc(apTweedy(s, x)))`` with ``dc`` = CG(n_iter) | one gradient step | identity:
    one library call forward, one backward (``csrc/adapt_ops.cu``).  The reverse sweep differentiates the unrolled
    CG recurrences exactly, as autograd does for the reference (src/samplers/utils.py:241-260)."""

    @staticmethod
    def forward(ctx, s, x, t, atb, y, rt, abar, gamma, n_iter, dc_code, lam, wts):
        import ctypes as C
        from .. import _lib
        lib = _lib.load()
        x = rt._prep(x, rt.im_shape, 'adapt x')
        s = rt._prep(s, rt.im_shape, 'adapt s')
        if s.shape != x.shape:
            raise ValueError('adapt: s %r and x %r differ in shape' % (tuple(s.shape), tuple(x.shape)))
        dev = x.device
        h = rt._handle(dev)
        batch = int(x.numel() // (rt.im_shape[0] * rt.im_shape[1]))
        atb = rt._prep(atb.to(dev).expand_as(x), rt.im_shape, 'adapt rhs') if atb is not None else None
        y = rt._prep(y.to(device=dev, dtype=torch.float32).expand(*x.shape[:-2], *rt.obs_shape), rt.obs_shape, 'adapt y')
        t = t.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        if t.numel() != batch:
            raise ValueError('adapt: one time step per sample expected')
        n_work = int(lib.scd_adapt_workspace_bytes(h.ptr, batch, int(n_iter)))
        work = torch.empty(n_work + 256, dtype=torch.uint8, device=dev)      # carries the saved vectors to backward
        wp = work.data_ptr() + (-work.data_ptr()) % 256
        loss = torch.empty((), dtype=torch.float32, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        w_user = wts.expanded(x.shape[:-2]).data_ptr() if wts is not None else None
        w_il = wts.packed(x.shape[:-2], dev) if wts is not None else None
        with torch.cuda.device(dev):
            _lib.check(lib.scd_adapt_fwd_w(h.ptr, x.data_ptr(), s.data_ptr(), atb.data_ptr() if atb is not None else None,
                                           y.data_ptr(), w_user, w_il, t.data_ptr(), abar.data_ptr(), int(abar.numel()),
                                           float(gamma), int(n_iter), int(dc_code), float(lam), loss.data_ptr(), None, batch,
                                           wp, n_work, stream), 'scd_adapt_fwd_w')
        ctx.rt, ctx.work, ctx.wp, ctx.n_work, ctx.batch, ctx.w_il = rt, work, wp, n_work, batch, w_il
        ctx.t, ctx.abar = t, abar
        ctx.args = (float(gamma), int(n_iter), int(dc_code), float(lam))
        ctx.shape = s.shape
        return loss

    @staticmethod
    def backward(ctx, g):
        import ctypes as C
        from .. import _lib
        lib = _lib.load()
        rt = ctx.rt
        if ctx.work is None:
            raise RuntimeError('the adaptation objective was already differentiated: its saved state lives in a workspace '
                               'that is released by the first backward pass (retain_graph is not supported)')
        dev = ctx.t.device
        h = rt._handle(dev)
        gamma, n_iter, dc_code, lam = ctx.args
        grad_s = torch.empty(ctx.shape, dtype=torch.float32, device=dev)
        g = g.to(device=dev, dtype=torch.float32).contiguous()
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with torch.cuda.device(dev):
            _lib.check(lib.scd_adapt_bwd_w(h.ptr, g.data_ptr(), ctx.w_il, ctx.t.data_ptr(), ctx.abar.data_ptr(),
                                           int(ctx.abar.numel()),
                                           # dx^2/ds: the mean cell cancels; the call backprojects without view weights
                                           gamma, n_iter, dc_code, lam, rt.adj_scale / rt.geometry.range_weight,
                                           grad_s.data_ptr(), ctx.batch, ctx.wp, ctx.n_work, stream), 'scd_adapt_bwd_w')
        ctx.work = None
        return (grad_s,) + (None,) * 11


def adapt_objective_applies(x, rhs, loss_fn, sde, dc_type: str) -> bool:
    """Whether the fused objective covers this call: :class:`AdaptationLoss` on a :class:`B200RayTrafo`, DDPM
    schedule, CUDA fp32, 4-D single-channel tensors, only the score output requiring grad."""
    from ..physics.b200_ray_trafo import B200RayTrafo
    from ..utils.sde import DDPM
    if not isinstance(loss_fn, AdaptationLoss) or not isinstance(loss_fn.ray_trafo, B200RayTrafo) or not isinstance(sde, DDPM):
        return False
    if dc_type not in _DC_CODES or not (x.is_cuda and x.dtype == torch.float32):
        return False
    if x.requires_grad or (rhs is not None and rhs.requires_grad) or loss_fn.observation.requires_grad:
        return False
    return x.dim() == 4 and x.shape[1] == 1


def adapt_objective(s, x, time_step, rhs, loss_fn: 'AdaptationLoss', sde, gamma: float, n_iter: int, dc_type: str):
    """Fused SCD adaptation objective, or ``None`` when the fused path does not apply (then the caller evaluates
    the reference's tensor expression)."""
    if not adapt_objective_applies(x, rhs, loss_fn, sde, dc_type) or s.shape != x.shape or s.dtype != torch.float32:
        return None
    return _AdaptObjectiveFn.apply(s, x, time_step, rhs, loss_fn.observation, loss_fn.ray_trafo,
                                   sde.alpha_bar_table(x.device), float(gamma), int(n_iter), _DC_CODES[dc_type],
                                   loss_fn.tv_penalty, loss_fn.weights)


def _score_model_adpt(score: nn.Module, impl: str = 'full', adpt_kwargs: Optional[Dict] = None,
                      verbose: bool = True, inject_fn=None) -> None:
    """Select the trainable parameters of the score model (reference :14-52).

    ``impl='lora'`` needs the LoRA injector of the caller's model package (the
    guided-diffusion UNet and its LoRA wrappers stay PyTorch code outside this
    package): pass it as ``inject_fn`` or run inside the reference checkout, where
    ``src.third_party_models.inject_trainable_lora_extended`` is importable."""
    score.requires_grad_(False)
    if impl == 'full':
        score.requires_grad_(True)
    elif impl == 'decoder':
        for part in (score.out, score.output_blocks):
            for name, param in part.named_parameters():
                if "emb_layers" not in name:
                    param.requires_grad = True
    elif impl == 'lora':
        for name, param in score.named_parameters():
            if "bias" in name and "emb_layers" not in name:
                param.requires_grad = True
        if inject_fn is None:
            try:
                from src.third_party_models import inject_trainable_lora_extended as inject_fn
            except ImportError as e:
                raise RuntimeError(
                    "impl='lora' needs a LoRA injector: pass inject_fn=... "
                    "(e.g. the reference's inject_trainable_lora_extended)") from e
        inject_fn(score, **(adpt_kwargs or {}))
    else:
        raise NotImplementedError(impl)

    if verbose:
        num_params = sum(p.numel() for p in score.parameters())
        trainable = sum(p.numel() for p in score.parameters() if p.requires_grad)
        print(f'% of trainable params: {trainable / num_params * 100}')
