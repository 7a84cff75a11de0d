"""Float64 oracle of the matched adjoint (helper module of the tests, not a test file).

The matched A* is the exact transpose of the Joseph projector: with ``c_w = dphi*ds/dx^2``, the Joseph matrix ``J``
of the oracle and the view weights ``w``,

    A* y = (adj_scale/dphi) * c_w * J^T diag(w) y
         = adj_scale * sum_i w_i sum_j k_i max(0, 1 - k_i |j - v_i|) y_ij,     k_i = 1 / max(|ci|, |si|)

(``v_i = ci*k0 + si*k1 + oi`` is the pixel's detector coordinate of the pixel-driven backprojector).
:func:`bp_hat64` restates the second line as the kernel evaluates it: two taps ``floor(v), floor(v)+1`` where
``h_i = 1/k_i <= 1``, three taps ``round(v)-1 .. round(v)+1`` where ``h_i > 1``.  :func:`bp64` is the first line.
The CG / DDS step in float64 repeat tests/fp64_reference.py on ``(J, c_w J^T diag(w))``.

Oracle geometries are ``oracle.OracleGeometry`` objects, optionally carrying view weights ``.w`` (as built by
``angle_set_oracle.geometry``); without ``.w`` every view weighs 1.
"""
from math import pi

import numpy as np

from fp64_reference import ddim64, tweedie64
from oracle import oracle as O


def weights(og):
    return np.asarray(getattr(og, 'w', np.ones(og.n_angles)), dtype=np.float64)


def c_w(og):
    return og.dphi * og.ds / og.dx ** 2


def view_constants(og):
    """Per view ``(ci, si, oi)`` of the backprojector (geometry.cu), float64 arrays."""
    c, s = np.cos(og.angles), np.sin(og.angles)
    ci = og.dx * c / og.ds
    si = og.dx * s / og.ds
    oi = ((og.x_min + 0.5 * og.dx) * c + (og.y_min + 0.5 * og.dx) * s - og.s_min) / og.ds - 0.5
    return ci, si, oi


def three_tap_views(og):
    """Boolean mask of the views whose hat is wider than one bin (``max(|ci|, |si|) > 1``)."""
    ci, si, _ = view_constants(og)
    return np.maximum(np.abs(ci), np.abs(si)) > 1.0


def bp_hat64(og, sino, rows=None):
    """The kernel's arithmetic in float64: ``adj_scale * sum_i w_i sum_taps k_i max(0, 1 - k_i |j - v|) y_ij``.
    ``rows``: only these image rows (index array), e.g. a sample of the rows of a large image."""
    y = np.asarray(sino, dtype=np.float64)
    lead = y.shape[:-2]
    y = y.reshape(-1, og.n_angles, og.n_det)
    rows = np.arange(og.n0) if rows is None else np.asarray(rows)
    k0 = rows.astype(np.float64)[:, None]
    k1 = np.arange(og.n1, dtype=np.float64)[None, :]
    ci, si, oi = view_constants(og)
    w = weights(og)
    out = np.zeros((y.shape[0], rows.size, og.n1))
    for i in range(og.n_angles):
        v = ci[i] * k0 + si[i] * k1 + oi[i]
        h = max(abs(ci[i]), abs(si[i]))
        k = 1.0 / h
        if h > 1.0:
            r = np.floor(v + 0.5).astype(np.int64)
            taps = (r - 1, r, r + 1)
        else:
            r = np.floor(v).astype(np.int64)
            taps = (r, r + 1)
        for j in taps:
            wt = k * np.maximum(0.0, 1.0 - k * np.abs(j - v))
            ok = (j >= 0) & (j < og.n_det)
            vals = np.zeros((y.shape[0],) + v.shape)
            vals[:, ok] = y[:, i, j[ok]] * wt[ok]
            out += w[i] * vals
    return (og.adj_scale * out).reshape(*lead, rows.size, og.n1)


_J = {}


def joseph(og):
    """The oracle's Joseph matrix (float64 CSR), cached per shape and angle list."""
    key = (og.im_shape, og.angles.tobytes())
    if key not in _J:
        _J[key] = O.joseph_matrix(og)
    return _J[key]


def bp_matrix(og):
    """The matched A* as a float64 CSR matrix ``(adj_scale/dphi) c_w J^T diag(w)``."""
    import scipy.sparse as sp
    J = joseph(og)
    return ((og.adj_scale / og.dphi) * c_w(og) * (J.T @ sp.diags(np.repeat(weights(og), og.n_det)))).tocsr()


def _cols(a, n):
    return np.asarray(a, dtype=np.float64).reshape(-1, n).T


def bp64(og, sino):
    """The matched A* of a batch of sinograms through the transposed Joseph matrix, float64."""
    y = np.asarray(sino, dtype=np.float64)
    lead = y.shape[:-2]
    cols = _cols(y, og.n_angles * og.n_det) * np.repeat(weights(og), og.n_det)[:, None]
    out = (og.adj_scale / og.dphi) * c_w(og) * (joseph(og).T @ cols)
    return out.T.reshape(*lead, og.n0, og.n1)


def fp64(og, img):
    x = np.asarray(img, dtype=np.float64)
    lead = x.shape[:-2]
    return (joseph(og) @ _cols(x, og.n0 * og.n1)).T.reshape(*lead, og.n_angles, og.n_det)


def normal64(og, v, gamma, add_identity=True):
    """``v + gamma A*(A v)`` with the matched A*, float64."""
    out = gamma * bp64(og, fp64(og, v))
    return out + np.asarray(v, dtype=np.float64) if add_identity else out


def cg64(og, x0, rhs, gamma, n_iter):
    """The reference's ``cg`` on ``(I + gamma A*A) x = rhs`` with the matched A*, per sample, float64."""
    J, Bm = joseph(og), bp_matrix(og)
    n = og.n0 * og.n1
    shape = np.shape(x0)
    op = lambda v: v + gamma * (Bm @ (J @ v))            # noqa: E731
    x = _cols(x0, n)
    with np.errstate(invalid='ignore', divide='ignore'):
        r = _cols(rhs, n) - op(x)
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
    return x.T.reshape(shape)


def dds_step64(og, x, s, atb, eps, t, t_prev, abar, gamma, eta, n_iter):
    """One DDS data-consistency step in float64 with the matched A*: ``(x_next, xhat0)``."""
    xhat0 = tweedie64(x, s, t, abar)
    atb = np.broadcast_to(np.asarray(atb, dtype=np.float64), xhat0.shape)
    xhat = cg64(og, xhat0, xhat0 + gamma * atb, gamma, n_iter) if n_iter > 0 else xhat0
    return ddim64(xhat, s, eps, t, t_prev, abar, eta), xhat0


def fbp64(og, sino):
    """FBP with the matched backprojector, float64: ``(dphi/dx^2) J^T diag(w) r`` with ``r`` the rows filtered by the
    reference recipe over ``pi/N_theta`` (see angle_set_oracle.fbp); on the uniform partition of [0, pi) this is
    ``J^T filter_sinogram(y) / dx^2``."""
    y = np.asarray(sino, dtype=np.float64)
    lead = y.shape[:-2]
    r = O.filter_sinogram(y) / (pi / og.n_angles)
    cols = _cols(r, og.n_angles * og.n_det) * np.repeat(weights(og), og.n_det)[:, None]
    out = (og.dphi / og.dx ** 2) * (joseph(og).T @ cols)
    return out.T.reshape(*lead, og.n0, og.n1)
