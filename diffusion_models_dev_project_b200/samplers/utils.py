"""Predictors and update rules of the DDS / SCD reverse sampler.

Call signatures follow reference src/samplers/utils.py (``:159-218`` DDS
predictor, ``:220-260`` ``_adapt``, ``:280-336`` adapted predictor, ``:338-368``
``ddim``, ``:370-378`` ``apTweedy``, ``:403-434`` schedule helpers), so that
``functools.partial`` objects and ``sample_kwargs['predictor']`` dictionaries
built for the reference work unchanged.

Dispatch rule (no silent fallbacks): with a :class:`B200RayTrafo`, a ``DDPM``
schedule, CUDA fp32 tensors and no gradient required, the work after the score
call runs in the fused sm_100a kernels; whenever a gradient is required (SCD
adaptation) or the schedule is VE/VP, the same formulas run as tensor
operations, with A / A* still executed by the CUDA projector kernels through
their autograd Functions.
"""
import os
from typing import Dict, Optional, Tuple, Union

import torch
from torch import Tensor

from .. import fused
from .adaptation import adapt_objective, adapt_objective_applies
from ..physics.b200_ray_trafo import B200RayTrafo, NormalOp, MeasurementWeights, as_weights
from ..utils.cg import cg
from ..utils.sde import SDE, VESDE, VPSDE, DDPM, _SCORE_PRED_CLASSES


# --------------------------------------------------------------- helpers ----
def _eps_pred_from_s(s, std_t):
    """Score-matching output -> epsilon prediction (reference :396-400)."""
    return - std_t * s


def _fusable(sde, *tensors) -> bool:
    if not isinstance(sde, DDPM):
        return False
    for t in tensors:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float32):
            return False
        if torch.is_grad_enabled() and t.requires_grad:
            return False
    return True


def _make_op(ray_trafo, gamma, weights=None):
    """``v + gamma A*(A v)``, or ``v + gamma A*(W A v)`` with measurement weights."""
    if isinstance(ray_trafo, B200RayTrafo):
        return NormalOp(ray_trafo, gamma, weights)
    if weights is not None:
        return lambda v: v + gamma * ray_trafo.trafo_adjoint(weights * ray_trafo(v))
    return lambda v: v + gamma * ray_trafo.trafo_adjoint(ray_trafo(v))


def _dc_weights(ray_trafo, cg_kwargs):
    """The measurement weights of the data consistency, ``cg_kwargs['weights']`` (None without).  Pass a
    :class:`MeasurementWeights` (the factories do): a plain tensor is validated and packed on every call."""
    weights = (cg_kwargs or {}).get('weights')
    if weights is not None and isinstance(ray_trafo, B200RayTrafo):
        weights = as_weights(ray_trafo, weights)
    return weights


def _weighted_gd(ray_trafo, xhat0, gamma, rhs, weights):
    """One gradient step on the data term: ``xhat0 - gamma A*(W A xhat0) + gamma rhs`` (W = 1 without weights)."""
    ax = ray_trafo(xhat0)
    if weights is not None:
        ax = (weights.w if isinstance(weights, MeasurementWeights) else weights) * ax
    return xhat0 - gamma * ray_trafo.trafo_adjoint(ax) + gamma * rhs


def apTweedy(s: Tensor, x: Tensor, sde: SDE, time_step: Tensor) -> Tensor:
    """Tweedie denoised estimate ``xhat0 = (x - std_t*eps_hat)/mean_t`` (reference :370-378)."""
    if _fusable(sde, s, x):
        return fused.tweedie_rhs(x, s, time_step, sde.alpha_bar_table(x.device))
    div = sde.marginal_prob_mean(time_step)[:, None, None, None].pow(-1)
    std_t = sde.marginal_prob_std(time_step)[:, None, None, None]
    if any(isinstance(sde, c) for c in _SCORE_PRED_CLASSES):
        s = _eps_pred_from_s(s=s, std_t=std_t)
    return (x - s * std_t) * div


def ddim(sde: SDE, s: Tensor, xhat: Tensor, time_step: Union[Tensor, Tuple[Tensor, Tensor]],
         step_size: Tensor, eta: float, use_simplified_eqn: bool = False) -> Tensor:
    """DDIM update (reference :338-368); VE, VP and DDPM branches."""
    pair = isinstance(time_step, tuple)
    t = time_step[0] if pair else time_step
    tminus1 = time_step[1] if pair else time_step - step_size
    if _fusable(sde, s, xhat):
        return fused.ddim_ddpm(xhat, s, torch.randn_like(xhat), t, tminus1,
                               sde.alpha_bar_table(xhat.device), eta)
    std_t = sde.marginal_prob_std(t=t)[:, None, None, None]
    if isinstance(sde, VESDE):
        std_tminus1 = sde.marginal_prob_std(t=tminus1)[:, None, None, None]
        tbeta = 1 - (std_tminus1.pow(2) * std_t.pow(-2)) if not use_simplified_eqn else torch.tensor(1.)
        noise_deterministic = - std_tminus1 * std_t * torch.sqrt(1 - tbeta.pow(2) * eta ** 2) * s
        noise_stochastic = std_tminus1 * eta * tbeta * torch.randn_like(xhat)
    elif isinstance(sde, (VPSDE, DDPM)):
        mean_tminus1 = sde.marginal_prob_mean(t=tminus1)[:, None, None, None]
        mean_t = sde.marginal_prob_mean(t=t)[:, None, None, None]
        tbeta = ((1 - mean_tminus1.pow(2)) / (1 - mean_t.pow(2))).pow(.5) * \
            (1 - mean_t.pow(2) * mean_tminus1.pow(-2)).pow(.5)
        # per-sample NaN -> 0 (the reference zeroes the whole batch if any entry is
        # NaN, :360; identical whenever all samples share the time step) -- no host sync
        tbeta = torch.nan_to_num(tbeta, nan=0.0, posinf=float('inf'), neginf=float('-inf'))
        xhat = xhat * mean_tminus1
        eps_ = _eps_pred_from_s(s, std_t) if isinstance(sde, VPSDE) else s
        noise_deterministic = torch.sqrt(1 - mean_tminus1.pow(2) - tbeta.pow(2) * eta ** 2) * eps_
        noise_stochastic = eta * tbeta * torch.randn_like(xhat)
    else:
        raise NotImplementedError
    return xhat + noise_deterministic + noise_stochastic


# ------------------------------------------------------------ predictors ----
def decomposed_diffusion_sampling_sde_predictor(
        score, sde: SDE, x: Tensor, rhs: Tensor,
        time_step: Union[Tensor, Tuple[Tensor, Tensor]],
        eta: float, gamma: float, step_size: float, cg_kwargs: Dict,
        datafitscale: Optional[float] = None,  # unused, kept for the call contract
        use_simplified_eqn: bool = False, ray_trafo=None) -> Tuple[Tensor, Tensor]:
    """Decomposed diffusion sampling step: score -> Tweedie -> CG data consistency
    on ``(I + gamma A*A) x = xhat0 + gamma A*y`` -> DDIM.  Returns ``(x_next, xhat0)``
    -- the second value is the Tweedie estimate, not the CG result (reference :218).
    ``cg_kwargs['weights']`` (optional measurement weights W, :class:`MeasurementWeights` or a tensor): CG on
    ``(I + gamma A*WA)``; ``rhs`` is then ``A*(W y)``.  (They ride in the solver options so that the predictor keeps
    the reference's signature.)"""
    weights = _dc_weights(ray_trafo, cg_kwargs)
    pair = isinstance(time_step, tuple)
    t = time_step[0] if pair else time_step
    with torch.no_grad():
        s = score(x, t)
        if pair and isinstance(ray_trafo, B200RayTrafo) and _fusable(sde, s, x, rhs):
            eps = torch.randn_like(x)
            x_next, xhat0 = ray_trafo.dds_step(
                x, s, rhs, eps, t, time_step[1], sde.alpha_bar_table(x.device),
                gamma=gamma, eta=eta, n_iter=cg_kwargs['max_iter'], weights=weights)
            return x_next.detach(), xhat0.detach()
        op = _make_op(ray_trafo, gamma, weights)
        xhat0 = apTweedy(s=s, x=x, sde=sde, time_step=t)
        xhat = cg(op=op, x=xhat0, rhs=xhat0 + gamma * rhs, n_iter=cg_kwargs['max_iter'])
        x = ddim(sde=sde, s=s, xhat=xhat, time_step=time_step, step_size=step_size, eta=eta,
                 use_simplified_eqn=use_simplified_eqn)
    return x.detach(), xhat0.detach()


_LORA_CLASSES = ('LoraInjectedLinear', 'LoraInjectedConv2d', 'LoraInjectedConv1d')


def _lora_modules(score):
    return [m for m in score.modules() if m.__class__.__name__ in _LORA_CLASSES]


def _tune_lora_scale(score, scale: float = 1.0):
    for m in _lora_modules(score):
        m.scale = scale


def _has_lora(score):
    return True if _lora_modules(score) else None


def _has_lora_active(score):
    mods = _lora_modules(score)
    return (mods[0].scale != 0) if mods else None


class _AdaptGraph:
    """One Adam step of :func:`_adapt` -- score call, fused adaptation objective (``scd_adapt_fwd`` /
    ``scd_adapt_bwd``), backward through the score model, optimizer step -- captured once in a CUDA graph and
    replayed ``num_steps`` times per reverse step.  The reference builds a fresh ``Adam`` for every reverse step
    (src/samplers/utils.py:240); the same effect is obtained by zeroing the moments and the step counter of the
    captured (``capturable=True``) optimizer before the replays.  Inputs live in static buffers."""

    def __init__(self, score, sde, loss_fn, x, time_step, rhs, lr, gamma, n_iter, dc_type):
        self.key = self.make_key(loss_fn, x, rhs, lr, gamma, n_iter, dc_type)
        self.x, self.t = x.detach().clone(), time_step.detach().clone()
        self.rhs = rhs.detach().clone() if rhs is not None else None
        params = list(score.parameters())
        self.optim = torch.optim.Adam(params, lr=lr, capturable=True)

        def one_step():
            s = score(self.x, self.t)
            loss = adapt_objective(s, self.x, self.t, self.rhs, loss_fn, sde, gamma, n_iter, dc_type)
            loss.backward()
            self.optim.step()
        # warm-up on a side stream (lazy optimizer state, library handles, kernel attributes), then undo it
        saved = [p.detach().clone() for p in params]
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):
            for _ in range(2):
                self.optim.zero_grad(set_to_none=True)
                one_step()
        torch.cuda.current_stream(x.device).wait_stream(side)
        with torch.no_grad():
            for p, q in zip(params, saved):
                p.copy_(q)
        self.reset()
        self.optim.zero_grad(set_to_none=True)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            one_step()

    @staticmethod
    def make_key(loss_fn, x, rhs, lr, gamma, n_iter, dc_type):
        # the captured graph holds the observation by address: a loss object that is re-used with another
        # observation (or an address recycled after garbage collection) must not hit a stale graph
        obs = loss_fn.observation
        # likewise the measurement weights (their packed copies are addressed by the graph)
        wts = getattr(loss_fn, 'weights', None)
        wkey = None if wts is None else (id(wts), wts.w.data_ptr(), wts.w._version)
        return (id(loss_fn), obs.data_ptr(), obs._version, tuple(obs.shape), loss_fn.tv_penalty, id(loss_fn.ray_trafo),
                tuple(x.shape), x.device, None if rhs is None else tuple(rhs.shape), float(lr), float(gamma), int(n_iter),
                dc_type, wkey)

    def reset(self):
        with torch.no_grad():
            for st in self.optim.state.values():
                st['exp_avg'].zero_(); st['exp_avg_sq'].zero_(); st['step'].zero_()

    def run(self, x, time_step, rhs, num_steps):
        self.x.copy_(x); self.t.copy_(time_step)
        if rhs is not None:
            self.rhs.copy_(rhs)
        self.reset()
        for _ in range(num_steps):
            self.graph.replay()


def _adapt(x: Tensor, score, sde: SDE, ray_trafo, loss_fn, time_step: Tensor, rhs: Tensor,
           num_steps: int, lr: float = 1e-3, gamma: float = 1e-3, n_iter: int = 1,
           dc_type: str = "cg", cuda_graph: Optional[bool] = None) -> None:
    """SCD adaptation: ``num_steps`` Adam steps on the trainable (LoRA / bias)
    parameters of ``score`` through Tweedie -> data consistency -> loss
    (reference :220-260).  Gradients flow through A, A* (CUDA kernels via their
    autograd Functions) and every CG recurrence.

    ``cuda_graph`` (default: environment variable ``SCD_ADAPT_CUDA_GRAPH=1``): capture one Adam step -- score
    model included -- in a CUDA graph and replay it (:class:`_AdaptGraph`); needs the fused objective (standard
    adaptation loss on the CUDA operator) and a score model that is safe to capture.

    Measurement weights ride on ``loss_fn`` (``AdaptationLoss(..., weights=W)``): the data-consistency step of the
    objective then solves ``(I + gamma A*WA)`` and ``rhs`` is ``A*(W y)``."""
    weights = getattr(loss_fn, 'weights', None)
    op = _make_op(ray_trafo, gamma, weights)
    assert _has_lora_active(score=score)
    score.eval()
    if cuda_graph is None:
        cuda_graph = os.environ.get('SCD_ADAPT_CUDA_GRAPH') == '1'
    if cuda_graph and adapt_objective_applies(x, rhs, loss_fn, sde, dc_type):
        g = getattr(score, '_scd_adapt_graph', None)
        key = _AdaptGraph.make_key(loss_fn, x, rhs, lr, gamma, n_iter, dc_type)
        if g is None or g.key != key:
            with torch.enable_grad():
                g = _AdaptGraph(score, sde, loss_fn, x, time_step, rhs, lr, gamma, n_iter, dc_type)
            object.__setattr__(score, '_scd_adapt_graph', g)
        g.run(x, time_step, rhs, num_steps)
        return
    optim = torch.optim.Adam(score.parameters(), lr=lr)
    for _ in range(num_steps):
        optim.zero_grad()
        s = score(x, time_step)
        # Tweedie -> data consistency -> loss and its whole backward sweep as two library calls when the loss is the
        # standard adaptation loss on the CUDA operator (same arithmetic as the tensor path below)
        loss = adapt_objective(s, x, time_step, rhs, loss_fn, sde, gamma, n_iter, dc_type) \
            if os.environ.get('SCD_ADAPT_UNFUSED') != '1' else None
        if loss is not None:
            loss.backward()
            optim.step()
            continue
        xhat0 = apTweedy(s=s, x=x, sde=sde, time_step=time_step)
        if dc_type == "cg":
            xhat = cg(op=op, x=xhat0, rhs=xhat0 + gamma * rhs, n_iter=n_iter)
        elif dc_type == "dc":
            xhat = _weighted_gd(ray_trafo, xhat0, gamma, rhs, weights)
        elif dc_type == "none":
            xhat = xhat0
        else:
            raise NotImplementedError
        loss = loss_fn(x=xhat)
        loss.backward()
        optim.step()


def adapted_ddim_sde_predictor(
        score, sde: SDE, x: Tensor, time_step: Union[Tensor, Tuple[Tensor, Tensor]],
        eta: float, step_size: float, adapt_fn, use_adapt: bool = False,
        datafitscale: Optional[float] = None, use_simplified_eqn: bool = False,
        ray_trafo=None, add_cg: bool = False, dc_type: str = None, gamma: float = None,
        cg_kwargs: Dict = None, rhs: Tensor = None) -> Tuple[Tensor, Tensor]:
    """SCD step (reference :280-336): optional adaptation, Tweedie with the adapted
    score, optional data consistency (``cg`` | ``gd`` | ``none``), DDIM with the
    un-adapted score (LoRA scale switched to 0 for that call).  ``cg_kwargs['weights']``: measurement weights W of
    the data consistency, ``(I + gamma A*WA)`` (``rhs`` is then ``A*(W y)``); the adaptation takes them from its
    loss."""
    weights = _dc_weights(ray_trafo, cg_kwargs)
    pair = isinstance(time_step, tuple)
    t = time_step[0] if pair else time_step
    if use_adapt:
        adapt_fn(x=x, time_step=t, ray_trafo=ray_trafo, rhs=rhs, gamma=gamma, n_iter=cg_kwargs['max_iter'])
    op = _make_op(ray_trafo, gamma, weights)
    with torch.no_grad():
        s = score(x, t)
        xhat0 = apTweedy(s=s, x=x, sde=sde, time_step=t)
        if add_cg:
            if dc_type == "cg":
                xhat = cg(op=op, x=xhat0, rhs=xhat0 + gamma * rhs, n_iter=cg_kwargs['max_iter'])
            elif dc_type == "gd":
                xhat = _weighted_gd(ray_trafo, xhat0, gamma, rhs, weights)
            elif dc_type == "none":
                xhat = xhat0
            else:
                raise NotImplementedError
        if _has_lora(score=score):
            _tune_lora_scale(score=score, scale=0)
        s = score(x, t)
        if _has_lora(score=score):
            _tune_lora_scale(score=score, scale=1.0)
        x = ddim(sde=sde, s=s, xhat=xhat if add_cg else xhat0, time_step=time_step,
                 step_size=step_size, eta=eta, use_simplified_eqn=use_simplified_eqn)
    return x.detach(), xhat0.detach()


def wrapper_ddim(score, sde: SDE, x: Tensor, time_step, step_size, datafitscale=1.):
    """Unconditional DDIM step with eta = 0.85 (reference :436-451)."""
    t = time_step[0] if isinstance(time_step, tuple) else time_step
    with torch.no_grad():
        s = score(x, t).detach()
        xhat0 = apTweedy(s=s, x=x, sde=sde, time_step=t)
        x = ddim(sde=sde, s=s, xhat=xhat0, time_step=time_step, step_size=step_size, eta=0.85,
                 use_simplified_eqn=False)
    return x.detach(), xhat0.detach()


# ---------------------------------- other guidance predictors (SURVEY 8f-4) ----
# Same boundary as the DDS path: the data-fit term is a callable on images that the drivers
# build from the ray transform (``nloglik = lambda x: norm(y - ray_trafo(x))``, reference
# src/utils/exp_utils.py:131,143,178); its gradient reaches A / A* through the autograd
# Functions of B200RayTrafo, i.e. the CUDA projector kernels.
def _datafit_grad(nloglik, at: Tensor, wrt: Tensor):
    loss = nloglik(at)
    return loss, torch.autograd.grad(outputs=loss, inputs=wrt)[0]


def Euler_Maruyama_sde_predictor(score, sde: SDE, x: Tensor, time_step: Tensor, step_size: float,
                                 nloglik: Optional[callable] = None, datafitscale: Optional[float] = None,
                                 penalty: Optional[float] = None, aTweedy: bool = False) -> Tuple[Tensor, Tensor]:
    """Reverse-SDE Euler-Maruyama step for VE / VP schedules (reference :11-67).

    ``aTweedy=False``: the data-fit gradient at ``x`` is subtracted from the score ("naive"
    guidance); ``aTweedy=True``: diffusion posterior sampling -- the data fit is evaluated at the
    Tweedie estimate, differentiated through the score model, scaled by ``1/loss`` and applied
    after the noise is added."""
    assert not isinstance(sde, DDPM)
    guided = nloglik is not None
    if guided:
        assert datafitscale is not None and penalty is not None
    x.requires_grad_()
    s = score(x, time_step)
    if not aTweedy:
        s = s.detach()
    grad = None
    if guided:
        target = apTweedy(s=s, x=x, sde=sde, time_step=time_step) if aTweedy else x
        loss, grad = _datafit_grad(nloglik, target, x)
        if aTweedy:
            datafitscale = loss.pow(-1)
    drift, diffusion = sde.sde(x, time_step)
    g2 = diffusion[:, None, None, None].pow(2)
    s_eff = s - penalty * grad * datafitscale if (guided and not aTweedy) else s
    x_mean = x - (drift - g2 * s_eff) * step_size
    x_new = x_mean + torch.sqrt(g2 * step_size) * torch.randn_like(x)
    if guided and aTweedy:
        x_new = x_new - penalty * grad * datafitscale
    return x_new.detach(), x_mean.detach()


def Ancestral_Sampling(score, sde: SDE, x: Tensor, time_step: Tuple[Tensor, Tensor], step_size: float,
                       nloglik: Optional[callable] = None, datafitscale: Optional[float] = None,
                       penalty: Optional[float] = None) -> Tuple[Tensor, Tensor]:
    """DDPM ancestral step with a fixed ``sigma_i = sqrt(1 - alpha_i)``; with ``nloglik`` it is DPS in
    the discrete framework (reference :70-125).  Returns ``(x_next, xhat0)``."""
    assert isinstance(sde, DDPM)
    t = time_step[0]
    guided = nloglik is not None
    if guided:
        assert penalty is not None
    with torch.set_grad_enabled(guided):
        if guided:
            x.requires_grad_()
        s = score(x, t)
        xhat0 = apTweedy(s=s, x=x, sde=sde, time_step=t)
        if guided:
            loss, grad = _datafit_grad(nloglik, xhat0, x)
            datafitscale = loss.pow(-1)
        std_t = sde.marginal_prob_std(t=t)[:, None, None, None]
        alpha_t = sde.alphas[int(t[0].item())]
        x_mean = 1 / torch.sqrt(alpha_t) * (x - (1 - alpha_t) / std_t * s)
        noise = torch.sqrt(1 - alpha_t) * torch.randn_like(x)
        if guided:
            x_mean = x_mean - penalty * grad * datafitscale
        x_new = x_mean + noise
    return x_new.detach(), xhat0.detach()


def Langevin_sde_corrector(score, sde: SDE, x: Tensor, time_step: Tensor, nloglik: Optional[callable] = None,
                           datafitscale: Optional[float] = None, penalty: Optional[float] = None,
                           corrector_steps: int = 1, snr: float = 0.16) -> Tensor:
    """Langevin MCMC corrector for VE / VP schedules (reference :128-157)."""
    assert not isinstance(sde, DDPM)
    guided = nloglik is not None
    if guided:
        assert datafitscale is not None and penalty is not None
    noise_norm = float(x[0].numel()) ** 0.5
    for _ in range(corrector_steps):
        x.requires_grad_()
        direction = score(x, time_step).detach()
        if guided:
            _, grad = _datafit_grad(nloglik, x, x)
            direction = direction - penalty * grad * datafitscale
        grad_norm = torch.norm(direction.reshape(direction.shape[0], -1), dim=-1).mean()
        eps = 2 * (snr * noise_norm / grad_norm) ** 2
        x = x + eps * direction + torch.sqrt(2 * eps) * torch.randn_like(x)
    return x.detach()


# -------------------------------------------------------------- schedule ----
def _check_times(times, t_0, num_steps):
    assert times[0] > times[1], (times[0], times[1])
    assert times[-1] == -1, times[-1]
    for t_last, t_cur in zip(times[:-1], times[1:]):
        assert abs(t_last - t_cur) == 1, (t_last, t_cur)
    for t in times:
        assert t >= t_0, (t, t_0)
        assert t <= num_steps, (t, num_steps)


def _schedule_jump(num_steps, travel_length, travel_repeat):
    """Time-travel schedule; ``[num_steps-1, ..., 0, -1]`` when length = repeat = 1
    (reference :416-434)."""
    jumps = {j: travel_repeat - 1 for j in range(0, num_steps - travel_length, travel_length)}
    t = num_steps
    time_steps = []
    while t >= 1:
        t -= 1
        time_steps.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] -= 1
            for _ in range(travel_length):
                t += 1
                time_steps.append(t)
    time_steps.append(-1)
    _check_times(time_steps, -1, num_steps)
    return time_steps
