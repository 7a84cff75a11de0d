"""Weighted oracle of limited-angle and non-uniform view sets (helper module of the tests, not a test file).

Built on the unchanged CPU oracle (oracle/oracle.py): an ``OracleGeometry`` whose angles and mean cell ``dphi`` are
those of a ``ParallelBeamGeometry2D``, plus the view weights ``w`` (ODL's relative angular cells).  A* with view
weights is the oracle's backprojector applied to the sinogram with row ``i`` scaled by ``w_i``:
``A* y = adj_scale * sum_i w_i lerp(y_i, t_i(x))``; its matrix is ``bp_matrix @ diag(w_i per detector bin)``.  A is
unweighted.  The float64 CG / DDS step repeats tests/fp64_reference.py on these matrices (cached per angle list and
weights) and reuses its Tweedie / DDIM restatements.
"""
from math import pi

import numpy as np

from fp64_reference import ddim64, tweedie64
from oracle import oracle as O


def geometry(geom, adj_scale=None, weighted=True):
    """The oracle geometry of a ``ParallelBeamGeometry2D``: its angles, mean cell ``dphi`` (default ``adj_scale``)
    and, as ``.w``, its view weights (ones when unweighted or ``weighted=False``)."""
    og = O.OracleGeometry(geom.im_shape, geom.n_angles)
    assert (og.n_det, og.s_min, og.ds, og.x_min, og.y_min, og.dx) == \
        (geom.n_det, geom.s_min, geom.ds, geom.x_min, geom.y_min, geom.dx)
    og.angles = np.array(geom.angles, dtype=np.float64)
    og.dphi = float(geom.dphi)
    og.adj_scale = og.dphi if adj_scale is None else float(adj_scale)
    w = geom.angle_weights if weighted else None
    og.w = np.ones(geom.n_angles) if w is None else np.array(w, dtype=np.float64)
    return og


def bp(og, sino):
    """Weighted A* with the C oracle: ``adj_scale * sum_i w_i lerp(sino_i)``."""
    y = np.asarray(sino, dtype=np.float64) * og.w[:, None]
    return O.bp(og, y.astype(np.float32))


def bp_matrix(og):
    """Weighted A* as a float64 CSR matrix (n0*n1, n_angles*n_det)."""
    import scipy.sparse as sp
    return (O.bp_matrix(og) @ sp.diags(np.repeat(og.w, og.n_det))).tocsr()


def fbp(og, sino):
    """FBP of any view set, float64: ``(dphi/ds) * sum_i w_i lerp(r_i, t_i(x))`` with ``r`` the rows filtered by
    the reference recipe (``O.filter_sinogram``) over ``pi/N_theta`` -- the recipe's constant ``pi/(2 N_theta)`` is
    ``2 pi/(2 N_theta)`` (the cell of the uniform partition of [0, pi)) times the 1/2 of its "2 Re" filter -- so
    that every view is summed with its own cell ``dphi * w_i``.  On the reference geometry this is ``O.fbp``; on a
    wedge it is the truncated FBP (the missing angles stay missing)."""
    y = np.asarray(sino, dtype=np.float64)
    q = O.filter_sinogram(y) / (pi / og.n_angles)
    lead = q.shape[:-2]
    q = q.reshape(-1, *og.obs_shape)
    x = og.x_min + (np.arange(og.n0) + 0.5) * og.dx
    yy = og.y_min + (np.arange(og.n1) + 0.5) * og.dx
    out = np.zeros((q.shape[0], og.n0 * og.n1))
    for i, phi in enumerate(og.angles):
        v = ((x[:, None] * np.cos(phi) + yy[None, :] * np.sin(phi)).ravel() - og.s_min) / og.ds - 0.5
        fl = np.floor(v); f = v - fl; j = fl.astype(np.int64)
        for jj, ww in ((j, 1.0 - f), (j + 1, f)):
            ok = (jj >= 0) & (jj < og.n_det)
            vals = np.zeros((q.shape[0], jj.size))
            vals[:, ok] = q[:, i, jj[ok]] * ww[ok]
            out += og.w[i] * vals
    out *= og.dphi / og.ds
    return out.reshape(*lead, *og.im_shape)


_MATRICES = {}


def matrices(og):
    """``(J, Bw)``: Joseph matrix and weighted A* in float64 CSR, cached per shape, scale, angles and weights."""
    key = (og.im_shape, og.adj_scale, og.angles.tobytes(), og.w.tobytes())
    m = _MATRICES.get(key)
    if m is None:
        m = _MATRICES[key] = (O.joseph_matrix(og), bp_matrix(og))
    return m


def cg64(og, x0, rhs, gamma, n_iter):
    """The reference's ``cg`` on ``(I + gamma A*A) x = rhs`` with the weighted A*, per sample, float64."""
    J, Bw = matrices(og)
    shape = np.shape(x0)
    cols = lambda a: np.asarray(a, dtype=np.float64).reshape(-1, og.n0 * og.n1).T      # noqa: E731
    op = lambda v: v + gamma * (Bw @ (J @ v))                                           # noqa: E731
    x = cols(x0)
    r = cols(rhs) - op(x)
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
    """One DDS data-consistency step in float64 with the weighted A*: ``(x_next, xhat0)``."""
    xhat0 = tweedie64(x, s, t, abar)
    atb = np.broadcast_to(np.asarray(atb, dtype=np.float64), xhat0.shape)
    xhat = cg64(og, xhat0, xhat0 + gamma * atb, gamma, n_iter) if n_iter > 0 else xhat0
    return ddim64(xhat, s, eps, t, t_prev, abar, eta), xhat0
