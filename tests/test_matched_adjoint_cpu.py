"""CPU tests of the matched adjoint: the kernel's arithmetic restated in float64 (two or three taps of the normalised
hat, split by the hat's half-width) is the exact transpose of the Joseph matrix on the reference geometries,
weighted view sets and views exactly on the axes; and the Python / C-ABI plumbing of ``adjoint='matched'``."""
import ctypes as C
from math import pi, sqrt
from types import SimpleNamespace as NS

import numpy as np
import pytest

import angle_set_oracle as W
import matched_adjoint_oracle as M
from conftest import rel_l2
from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D as G
from oracle import oracle as O


def _golden(n):
    return np.mod(np.arange(n) * pi * (3.0 - sqrt(5.0)), pi)


GEOMETRIES = {
    '256x256-60': lambda: G.from_im_shape((256, 256), 60),
    '96x70-18': lambda: G.from_im_shape((96, 70), 18),
    '501x501-40': lambda: G.from_im_shape((501, 501), 40),
    'wedge90': lambda: G.from_angle_range((256, 256), 60, 0.0, pi / 2),
    'golden37': lambda: G.from_angles((256, 256), _golden(37)),
    'axes': lambda: G.from_angles((96, 70), [0.0, pi / 4, pi / 2]),
}


@pytest.mark.parametrize('name', list(GEOMETRIES))
def test_hat_restatement_is_the_transpose_of_the_joseph_matrix(name):
    geom = GEOMETRIES[name]()
    og = W.geometry(geom)
    if name == 'golden37':
        assert geom.angle_weights is not None
    y = np.random.default_rng(3).standard_normal((2, *geom.obs_shape))
    got = M.bp_hat64(og, y)
    J = O.joseph_matrix(og)
    cw = geom.dphi * geom.ds / geom.dx ** 2
    ref = np.stack([cw * (J.T @ (y[b] * og.w[:, None]).ravel()).reshape(geom.im_shape) for b in range(2)])
    for b in range(2):
        assert rel_l2(got[b], ref[b]) <= 1e-12, (name, b, rel_l2(got[b], ref[b]))
    # and the matrix form the GPU tests use
    assert rel_l2(M.bp64(og, y), ref) <= 1e-12
    # the pixel-driven A* is far from it on white noise
    assert rel_l2(W.bp(og, y.astype(np.float32)), ref) > 1e-2


def test_three_tap_view_counts():
    counts = {name: int(M.three_tap_views(W.geometry(GEOMETRIES[name]())).sum())
              for name in ('256x256-60', '96x70-18', '501x501-40', 'axes')}
    assert counts == {'256x256-60': 8, '96x70-18': 4, '501x501-40': 4, 'axes': 2}
    # the hat never reaches a fourth bin: half-width <= dx/ds < 1.5 on every geometry SimpleTrafo derives
    for shape in ((256, 256), (501, 501), (96, 70), (70, 50), (24, 24)):
        g = G.from_im_shape(shape, 8)
        assert 1.0 < g.dx / g.ds < 1.5


def test_the_third_tap_is_needed():
    """Dropping the third tap of the near-axis views (using floor(v), floor(v)+1 everywhere) lands ~20x beyond the
    1e-5 gate of the GPU tests at 256^2 / 60 (the hat is only 0.8% wider than a bin there: about 1.9e-4)."""
    geom = GEOMETRIES['256x256-60']()
    og = W.geometry(geom)
    y = np.random.default_rng(5).standard_normal(geom.obs_shape)
    ref = M.bp64(og, y)
    ci, si, oi = M.view_constants(og)
    k0 = np.arange(og.n0)[:, None]
    k1 = np.arange(og.n1)[None, :]
    two = np.zeros(og.im_shape)
    for i in range(og.n_angles):
        v = ci[i] * k0 + si[i] * k1 + oi[i]
        k = 1.0 / max(abs(ci[i]), abs(si[i]))
        r = np.floor(v).astype(np.int64)
        for j in (r, r + 1):
            ok = (j >= 0) & (j < og.n_det)
            two[ok] += (k * np.maximum(0.0, 1.0 - k * np.abs(j - v)) * np.where(ok, y[i, np.clip(j, 0, og.n_det - 1)], 0))[ok]
    assert rel_l2(og.dphi * two, ref) > 1e-4


# ------------------------------------------------------------------------------------------------ plumbing ---
def test_adjoint_argument_is_validated():
    import diffusion_models_dev_project_b200 as pkg
    assert pkg.B200RayTrafo((32, 32), 6).adjoint == 'pixel'
    assert pkg.B200RayTrafo((32, 32), 6, adjoint='matched').adjoint == 'matched'
    for bad in ('Matched', 'exact', None, 1):
        with pytest.raises(ValueError):
            pkg.B200RayTrafo((32, 32), 6, adjoint=bad)


def test_sharded_operator_reports_the_base_setting():
    from diffusion_models_dev_project_b200 import B200RayTrafo
    from diffusion_models_dev_project_b200.sharding import AngleShardedRayTrafo
    assert AngleShardedRayTrafo(B200RayTrafo((32, 32), 6, adjoint='matched')).adjoint == 'matched'
    assert AngleShardedRayTrafo(B200RayTrafo((32, 32), 6)).adjoint == 'pixel'


def _config(**fo):
    return NS(forward_op=NS(trafo_name='simple_trafo', num_angles=12, impl='b200', **fo), data=NS(im_size=32))


def test_factory_reads_the_adjoint_key():
    import diffusion_models_dev_project_b200 as pkg
    assert pkg.get_standard_ray_trafo(_config()).adjoint == 'pixel'
    assert pkg.get_standard_ray_trafo(_config(adjoint='pixel')).adjoint == 'pixel'
    assert pkg.get_standard_ray_trafo(_config(adjoint='matched')).adjoint == 'matched'
    rt = pkg.get_standard_ray_trafo(_config(adjoint='matched', angle_range=(0.0, pi / 2)))
    assert rt.adjoint == 'matched' and rt.geometry.dphi == pytest.approx(pi / 24)
    rt = pkg.get_standard_ray_trafo(_config(adjoint='matched', angles=_golden(12)))
    assert rt.adjoint == 'matched' and rt.geometry.angle_weights is not None
    with pytest.raises(ValueError):
        pkg.get_standard_ray_trafo(_config(adjoint='exact'))


def test_binding_declares_scd_geom_create_ex():
    from diffusion_models_dev_project_b200 import _lib
    res, args = _lib.SIGNATURES['scd_geom_create_ex']
    assert res is C.c_int
    assert args == [C.POINTER(_lib.GeomDesc), C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_void_p)]
    assert _lib.SCD_GEOM_MATCHED_ADJOINT == 1


def _desc(dx, ds):
    ang = np.array([0.1, 0.2])
    d = _lib_mod().GeomDesc(n0=8, n1=8, x_min=-4 * dx, y_min=-4 * dx, dx=dx, n_angles=2,
                            angles=ang.ctypes.data_as(C.POINTER(C.c_double)), n_det=13, s_min=-6.5 * ds, ds=ds,
                            adj_scale=1)
    d._keep = ang
    return d


def _lib_mod():
    from diffusion_models_dev_project_b200 import _lib
    return _lib


@pytest.mark.parametrize('flags,dx,ds', [(0x2, 1.0, 1.0), (0x80000001, 1.0, 1.0), (1, 1.5, 1.0), (1, 3.0, 1.0)])
def test_geom_create_ex_rejects_before_touching_a_device(flags, dx, ds):
    """Unknown flag bits, and the matched adjoint on dx/ds >= 1.5, are rejected whether or not a GPU is present: the
    handle stays NULL."""
    _lib = _lib_mod()
    lib = _lib.load()
    d = _desc(dx, ds)
    h = C.c_void_p(12345)
    assert lib.scd_geom_create_ex(C.byref(d), None, flags, C.byref(h)) == _lib.SCD_E_INVALID
    assert not h.value
    assert ('unknown flag' in _lib.last_error()) if flags != 1 else ('dx/ds < 1.5' in _lib.last_error())
