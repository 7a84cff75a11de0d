"""Float64 reference of the fused DDS data-consistency step (helper module of the tests, not a test file).

The operators are the oracle's sparse restatements (oracle/oracle.py): the Joseph matrix ``J`` for A and the
pixel-driven backprojection matrix ``Bm`` for A* (it already carries ``adj_scale``), built once per geometry in
float64.  On them the step is evaluated as the reference writes it (src/samplers/utils.py:195-218):

  xhat0 = (x - s * sqrt(1 - abar_t)) / sqrt(abar_t)                     apTweedy      (:370-378)
  xhat  = cg((I + gamma A*A), x = xhat0, rhs = xhat0 + gamma * atb)      cg            (src/utils/cg.py:11-39)
  x'    = sqrt(abar_tp) xhat + sqrt(1 - abar_tp - tbeta^2 eta^2) s + eta tbeta eps     ddim, DDPM branch (:356-368)

with ``abar_t = abar[trunc(t) + 1]`` clamped to the table, as ``Tensor.long() + 1`` indexes it and as the kernels do
(``il_abar_at``, ``abar_at``).  The only inputs in float32 are the arguments themselves (and the values of the fp32
alpha-bar table); every operation after that is float64.
"""
import numpy as np

from oracle import oracle as O

_MATRICES = {}


def matrices(geom):
    """``(J, Bm)`` of ``geom`` in float64 CSR, cached per geometry."""
    key = (geom.im_shape, geom.n_angles, geom.adj_scale)
    m = _MATRICES.get(key)
    if m is None:
        m = (O.joseph_matrix(geom), O.bp_matrix(geom))
        _MATRICES[key] = m
    return m


def _columns(a, geom):
    """``[B, ..., n0, n1]`` -> float64 ``[n0*n1, B]`` (one sample per column)."""
    a = np.asarray(a, dtype=np.float64)
    return a.reshape(-1, geom.n0 * geom.n1).T


def cg64(geom, x0, rhs, gamma, n_iter):
    """The reference's ``cg`` on ``(I + gamma A*A) x = rhs`` from ``x0``, per sample, in float64.

    Fixed ``n_iter`` iterations and no guard against a zero residual, exactly like the kernels: a sample whose
    residual is exactly zero divides 0/0 and comes out NaN.  Returns float64 of ``x0``'s shape."""
    J, Bm = matrices(geom)
    shape = np.shape(x0)
    x = _columns(x0, geom)
    op = lambda v: v + gamma * (Bm @ (J @ v))            # noqa: E731
    with np.errstate(invalid='ignore', divide='ignore'):
        r = _columns(rhs, geom) - op(x)
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


def abar_at(abar, t):
    """``abar[trunc(t) + 1]`` clamped to the table, per sample (float64 values of the fp32 table)."""
    abar = np.asarray(abar, dtype=np.float64).reshape(-1)
    idx = np.trunc(np.asarray(t, dtype=np.float64).reshape(-1)).astype(np.int64) + 1
    return abar[np.clip(idx, 0, abar.size - 1)]


def _per_sample(v, shape):
    """One value per sample, shaped to broadcast against a ``shape`` batch."""
    return np.asarray(v, dtype=np.float64).reshape(shape[0], *([1] * (len(shape) - 1)))


def tweedie64(x, s, t, abar):
    """``apTweedy`` of the DDPM: ``(x - s sqrt(1 - abar_t)) / sqrt(abar_t)``, per-sample ``t``."""
    x = np.asarray(x, dtype=np.float64)
    ab = abar_at(abar, t)
    return (x - np.asarray(s, dtype=np.float64) * _per_sample(np.sqrt(1.0 - ab), x.shape)) / _per_sample(np.sqrt(ab), x.shape)


def ddim64(xhat, s, eps, t, t_prev, abar, eta):
    """DDPM branch of ``ddim`` with the noise ``eps`` passed in, per-sample ``(t, t_prev)``.

    A NaN ``tbeta`` (``t_prev`` later than ``t``: ``1 - abar_t/abar_tp < 0``) is set to 0 **per sample**, as the
    package's ``ddim`` and the kernels do.  The reference zeroes ``tbeta`` of the whole batch when any entry is NaN;
    the two rules agree whenever every sample has the same pair of time steps, and per sample when the reference
    is run one sample at a time."""
    xhat = np.asarray(xhat, dtype=np.float64)
    m_t, m_p = np.sqrt(abar_at(abar, t)), np.sqrt(abar_at(abar, t_prev))
    with np.errstate(invalid='ignore', divide='ignore'):
        tbeta = np.sqrt((1.0 - m_p ** 2) / (1.0 - m_t ** 2)) * np.sqrt(1.0 - m_t ** 2 / m_p ** 2)
    tbeta = np.where(np.isnan(tbeta), 0.0, tbeta)
    det = np.sqrt(1.0 - m_p ** 2 - tbeta ** 2 * eta ** 2)
    col = lambda v: _per_sample(v, xhat.shape)            # noqa: E731
    return (xhat * col(m_p) + col(det) * np.asarray(s, dtype=np.float64)
            + col(eta * tbeta) * np.asarray(eps, dtype=np.float64))


def dds_step64(geom, x, s, atb, eps, t, t_prev, abar, gamma, eta, n_iter):
    """One DDS data-consistency step in float64: returns ``(x_next, xhat0)``, both of ``x``'s shape.

    :func:`tweedie64`, then :func:`cg64` on ``(I + gamma A*A) x = xhat0 + gamma atb`` from ``xhat0``, then
    :func:`ddim64` (per-sample NaN rule for ``tbeta``, see there).  ``t`` and ``t_prev`` hold one time step per
    sample; ``atb`` has ``x``'s shape or broadcasts to it."""
    xhat0 = tweedie64(x, s, t, abar)
    atb = np.broadcast_to(np.asarray(atb, dtype=np.float64), xhat0.shape)
    xhat = cg64(geom, xhat0, xhat0 + gamma * atb, gamma, n_iter) if n_iter > 0 else xhat0
    return ddim64(xhat, s, eps, t, t_prev, abar, eta), xhat0


# ---- shared inputs of the tests --------------------------------------------------------------------------------
# (t, t_prev) of sample b is TIME_PAIRS[b % 8]: (250.6, 240) exercises the truncation of t, (0, -1) reaches
# abar[0] = 1, (100, 120) has a NaN tbeta (set to 0), the others are ordinary steps of a 1000-step schedule
TIME_PAIRS = ((999., 989.), (500., 490.), (250.6, 240.), (10., 0.), (0., -1.), (700., 690.), (100., 120.), (3., 2.))
BENCH_PAIR = (500., 490.)


def time_steps(batch, pairs=TIME_PAIRS):
    """float32 arrays ``(t, t_prev)`` of a batch: sample ``b`` takes ``pairs[b % len(pairs)]``."""
    tt = np.array([pairs[b % len(pairs)] for b in range(batch)], dtype=np.float32)
    return tt[:, 0].copy(), tt[:, 1].copy()


_PORT_TRAFOS = {}


def port_trafo(geom):
    """The oracle's float32 ray trafo of ``geom`` (cached), for the ``O.ref_port_*`` functions.  Its two matrices
    are stored as CSR instead of COO: the same float32 entries, but one product on the CPU takes milliseconds
    instead of ~0.4 s."""
    key = (geom.im_shape, geom.n_angles, geom.adj_scale)
    rt = _PORT_TRAFOS.get(key)
    if rt is None:
        rt = O.OracleRayTrafo(geom)
        rt.matrix = rt.matrix.to_sparse_csr()
        rt.matrix_adj = rt.matrix_adj.to_sparse_csr()
        _PORT_TRAFOS[key] = rt
    return rt


def port_dds_step(geom, x, s, atb, eps, t, t_prev, abar, gamma, eta, n_iter):
    """``O.ref_port_dds_step`` -- the float32 port of the reference's predictor body -- run one sample at a time
    (where the reference's batch-wide NaN rule for ``tbeta`` is the per-sample one).  numpy in, numpy out:
    ``(x_next, xhat0)``."""
    import torch
    rt = port_trafo(geom)
    ab = torch.as_tensor(np.asarray(abar, dtype=np.float32))
    f = lambda a, b: torch.from_numpy(np.ascontiguousarray(a[b:b + 1], dtype=np.float32))    # noqa: E731
    outs, xh0s = [], []
    for b in range(np.shape(x)[0]):
        sb = f(s, b)
        out, xh0 = O.ref_port_dds_step(lambda *_: sb, f(x, b), f(atb, b), ab, f(t, b), f(t_prev, b),
                                       gamma, eta, n_iter, rt, noise=f(eps, b))
        outs.append(out.numpy())
        xh0s.append(xh0.numpy())
    return np.concatenate(outs), np.concatenate(xh0s)
