"""Batched conjugate gradient for ``(I + gamma A*A) x = rhs``.

Signature of the reference's ``cg(op, x, rhs, n_iter, tol)``
(src/utils/cg.py:11-39): fixed ``n_iter`` iterations from the start value ``x``,
per-sample step sizes over dims [1,2,3], no tolerance test (``tol`` is accepted
and, as in the reference, unused) and no guard against a zero residual.

When ``op`` is a :class:`~..physics.b200_ray_trafo.NormalOp` on a
:class:`B200RayTrafo` and no gradient is required, the whole solve runs as the
fused CUDA launch sequence ``scd_cg`` (A, A* with the axpy and <p,d> in its
epilogue, one update kernel, one direction kernel per iteration); a ``NormalOp``
with measurement weights, ``v + gamma A*(W A v)``, takes the same path (``scd_cg_w``).  Any other
callable -- and every call that must be differentiated, e.g. the LoRA
adaptation of SCD (reference src/samplers/utils.py:241-260) -- runs the same
recurrences as tensor operations on whatever device the tensors live on.
"""
import torch
from torch import Tensor


def _fused_ok(op, x: Tensor, rhs: Tensor) -> bool:
    from ..physics.b200_ray_trafo import B200RayTrafo, NormalOp
    if not isinstance(op, NormalOp) or not isinstance(op.ray_trafo, B200RayTrafo):
        return False
    if torch.is_grad_enabled() and (x.requires_grad or rhs.requires_grad):
        return False
    return x.is_cuda and x.dtype == torch.float32 and x.dim() == 4


def _bdot(a, b):
    return (a * b).sum(dim=[1, 2, 3])


def _col(v):
    return v[:, None, None, None]


class _CgSelfAdjointFn(torch.autograd.Function):
    """The CG recurrences of :func:`cg` with a hand-written reverse sweep, for an operator whose
    vector-Jacobian product is the operator itself (``op_nograd(g)``).

    That holds for ``op(v) = v + gamma*A*(A v)`` on :class:`B200RayTrafo`: with ODL's gradient pairing
    (grad of ``trafo`` = ``A*(g)/c_w``, grad of ``trafo_adjoint`` = ``c_w*A(g)``, SURVEY.md 8b) the
    gradient through ``op`` is ``g + gamma*A*(A g)`` -- and ``g + gamma*A*(W A g)`` with measurement weights,
    a diagonal between the two.  The forward pass runs the same recurrences as the
    tensor path below (same values), keeps ``p_k, d_k, r_{k+1}`` and the scalars of every iteration, and
    the backward pass differentiates them exactly -- the iterates are a non-linear function of ``x`` and
    ``rhs`` (alpha, beta), so this is NOT the adjoint linear solve -- with ``n_iter + 1`` operator
    applications and no autograd graph over the ~25 tensor operations per iteration.  It is what the LoRA
    adaptation of SCD differentiates ten times per reverse step (reference src/samplers/utils.py:241-260).
    """

    @staticmethod
    def forward(ctx, x, rhs, op_nograd, n_iter):
        r = rhs - op_nograd(x)
        p = r
        rr = _bdot(r, r)
        saved, scal = [r], []
        for _ in range(n_iter):
            d = op_nograd(p)
            pd = _bdot(p, d)
            alpha = rr / pd
            x = x + _col(alpha) * p
            r = r - _col(alpha) * d
            rr_new = _bdot(r, r)
            beta = rr_new / rr
            saved += [p, d, r]
            scal.append((alpha, beta, rr, pd, rr_new))
            rr = rr_new
            p = r + _col(beta) * p
        ctx.op = op_nograd
        ctx.scal = scal
        ctx.n_iter = n_iter
        ctx.save_for_backward(*saved)
        return x

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        op = ctx.op
        r0 = saved[0]
        gx = g                                     # adjoint of x_{k+1}
        gr = torch.zeros_like(g)                   # adjoint of r_{k+1}
        gp = torch.zeros_like(g)                   # adjoint of p_{k+1}
        grho = torch.zeros_like(ctx.scal[0][0]) if ctx.n_iter else None     # adjoint of rho_{k+1}
        for k in range(ctx.n_iter - 1, -1, -1):
            p, d, r1 = saved[1 + 3 * k], saved[2 + 3 * k], saved[3 + 3 * k]
            alpha, beta, rho, pd, rho1 = ctx.scal[k]
            # p_{k+1} = r_{k+1} + beta_k p_k ;  beta_k = rho_{k+1}/rho_k ;  rho_{k+1} = <r_{k+1}, r_{k+1}>
            gbeta = _bdot(gp, p)
            grho1 = grho + gbeta / rho
            gr1 = gr + gp + _col(2.0 * grho1) * r1
            gp_k = _col(beta) * gp
            grho_k = -gbeta * beta / rho
            # r_{k+1} = r_k - alpha_k d_k ;  x_{k+1} = x_k + alpha_k p_k ;  alpha_k = rho_k / <p_k, d_k>
            galpha = _bdot(gx, p) - _bdot(gr1, d)
            gpd = -galpha * alpha / pd
            grho_k = grho_k + galpha / pd
            gd = _col(gpd) * p - _col(alpha) * gr1
            gp_k = gp_k + _col(alpha) * gx + _col(gpd) * d + op(gd)        # d_k = op(p_k), op self-adjoint
            gr, gp, grho = gr1, gp_k, grho_k
        # rho_0 = <r_0, r_0>, p_0 = r_0, r_0 = rhs - op(x_0)
        if ctx.n_iter:
            gr = gr + gp + _col(2.0 * grho) * r0
        grad_rhs = gr
        grad_x = gx - op(gr)
        return grad_x, grad_rhs, None, None


def _self_adjoint_nograd(op):
    """``op`` evaluated without recording a graph, when its gradient is known to be ``op`` itself."""
    from ..physics.b200_ray_trafo import B200RayTrafo, NormalOp
    if isinstance(op, NormalOp) and isinstance(op.ray_trafo, B200RayTrafo):
        rt, gamma, weights = op.ray_trafo, op.gamma, op.weights
        return lambda v: rt.normal_apply(v, gamma, weights=weights)
    return None


def cg(op: callable, x: Tensor, rhs: Tensor, n_iter: int = 5, tol: float = 1e-10) -> Tensor:
    if _fused_ok(op, x, rhs):
        return op.ray_trafo.cg_solve(x, rhs, op.gamma, n_iter, weights=op.weights)
    if torch.is_grad_enabled() and (x.requires_grad or rhs.requires_grad) and x.is_cuda and x.dim() == 4:
        op_nograd = _self_adjoint_nograd(op)
        if op_nograd is not None:
            return _CgSelfAdjointFn.apply(x, rhs, op_nograd, int(n_iter))

    bdot = _bdot
    r = rhs - op(x)
    p = r
    rr = bdot(r, r)
    for _ in range(n_iter):
        d = op(p)
        alpha = rr / bdot(p, d)
        x = x + alpha[:, None, None, None] * p
        r = r - alpha[:, None, None, None] * d
        rr_new = bdot(r, r)
        beta = rr_new / rr
        rr = rr_new
        p = r + beta[:, None, None, None] * p
    return x
