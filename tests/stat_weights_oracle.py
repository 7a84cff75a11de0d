"""Float64 oracle of the weighted data-consistency system (helper module of the tests, not a test file).

With measurement weights ``W`` (one per sample, view and bin) the operator of the DDS / SCD data consistency is

    op(v) = v + gamma * Bm @ (W * (J @ v))        (J: Joseph matrix = A,  Bm: matrix of A*, view weights included)

evaluated per sample (one column each).  ``J`` and ``Bm`` come from the existing restatements: the pixel-driven A*
with view weights of angle_set_oracle (ones on a uniform partition) or the matched A* of matched_adjoint_oracle.
The CG recurrences of tests/fp64_reference.py are restated once, on any operator of columns (:func:`cg_cols`): its
``cg64`` builds the unweighted operator inside and is kept unchanged as the yardstick the unweighted tests use (the
CPU tests check that :func:`cg64` with ``W = 1`` reproduces it).  The DDS step reuses its Tweedie / DDIM.
"""
import numpy as np

import angle_set_oracle as AO
import matched_adjoint_oracle as MO
from fp64_reference import ddim64, tweedie64


def matrices(og, adjoint='pixel'):
    """``(J, Bm)`` of an oracle geometry carrying view weights ``.w`` (angle_set_oracle.geometry)."""
    if adjoint == 'matched':
        return MO.joseph(og), MO.bp_matrix(og)
    return AO.matrices(og)


def _cols(a, n):
    return np.asarray(a, dtype=np.float64).reshape(-1, n).T


def weight_cols(og, w, batch):
    """``W`` (broadcastable to ``[batch, 1, n_angles, n_det]``) as float64 columns ``[n_angles*n_det, batch]``."""
    w = np.asarray(w, dtype=np.float64).reshape(-1, og.n_angles * og.n_det)
    return np.broadcast_to(w, (batch, w.shape[1])).T


def normal64(J, Bm, og, v, gamma, w, add_identity=True):
    """``v + gamma A*(W A v)`` per sample, float64, of ``v``'s shape."""
    n = og.n0 * og.n1
    shape = np.shape(v)
    vc = _cols(v, n)
    out = gamma * (Bm @ (weight_cols(og, w, vc.shape[1]) * (J @ vc)))
    return (out + vc if add_identity else out).T.reshape(shape)


def cg_cols(op, x, rhs, n_iter):
    """The reference's ``cg`` (src/utils/cg.py:11-39) on float64 columns (one sample each) for the operator ``op`` of
    columns: fixed ``n_iter`` iterations, no guard against a zero residual."""
    with np.errstate(invalid='ignore', divide='ignore'):
        r = rhs - op(x)
        p = r.copy()
        rr = (r * r).sum(0)
        for _ in range(int(n_iter)):
            d = op(p)
            alpha = rr / (p * d).sum(0)
            x = x + alpha * p
            r = r - alpha * d
            rr_new = (r * r).sum(0)
            p = r + (rr_new / rr) * p
            rr = rr_new
    return x


def cg64(J, Bm, og, x0, rhs, gamma, n_iter, w):
    """The reference's ``cg`` on ``(I + gamma A*WA) x = rhs`` from ``x0``, per sample, float64."""
    n = og.n0 * og.n1
    x = _cols(x0, n)
    wc = weight_cols(og, w, x.shape[1])
    op = lambda v: v + gamma * (Bm @ (wc * (J @ v)))      # noqa: E731
    return cg_cols(op, x, _cols(rhs, n), n_iter).T.reshape(np.shape(x0))


def dds_step64(J, Bm, og, x, s, atb, eps, t, t_prev, abar, gamma, eta, n_iter, w):
    """One weighted DDS step in float64 (``atb`` = A*(W y)): ``(x_next, xhat0)``."""
    xhat0 = tweedie64(x, s, t, abar)
    atb = np.broadcast_to(np.asarray(atb, dtype=np.float64), xhat0.shape)
    xhat = cg64(J, Bm, og, xhat0, xhat0 + gamma * atb, gamma, n_iter, w) if n_iter > 0 else xhat0
    return ddim64(xhat, s, eps, t, t_prev, abar, eta), xhat0


def poisson64(ax, photons, mu, rng, min_count=0.1):
    """numpy restatement of ``simulate_poisson`` on a float32 projection ``ax``: ``(counts, y, W)``."""
    lam = photons * np.exp(-mu * np.asarray(ax, dtype=np.float64))
    counts = np.maximum(rng.poisson(lam), min_count)
    y = -np.log(counts / photons) / mu
    w = counts / counts.reshape(counts.shape[0], -1).mean(axis=1).reshape(-1, *([1] * (counts.ndim - 1)))
    return counts, y, w
