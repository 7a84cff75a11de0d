"""CPU tests of limited-angle and non-uniform view sets: the host geometry (``from_angle_range``,
``from_angles`` and their view weights) and the weighted oracle (A*, bp_matrix, FBP) the GPU tests compare
against."""
from math import ceil, pi, sqrt

import numpy as np
import pytest

import angle_set_oracle as W
from bench_support.phantoms import disk_ellipses
from conftest import rel_l2
from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D as G
from oracle import oracle as O


def _golden_angles(n):
    return np.mod(np.arange(n) * pi * (3.0 - sqrt(5.0)), pi)


# ---------------------------------------------------------------------------------------------- geometry ---
@pytest.mark.parametrize('im_shape,na', [((256, 256), 60), ((501, 501), 1200), ((96, 70), 18)])
def test_from_im_shape_is_unchanged(im_shape, na):
    g = G.from_im_shape(im_shape, na)
    # the rule of SimpleTrafo.__init__ (SURVEY.md §3.5), written out independently of the class
    n0, n1 = im_shape
    lo = ((-n0) // 2, (-n1) // 2)
    dx = (n0 // 2 - lo[0]) / n0
    rho = max(sqrt(x * x + y * y) for x in (lo[0], n0 // 2) for y in (lo[1], n1 // 2))
    n_det = 2 * int(ceil(rho / dx)) + 1
    assert (g.n0, g.n1, g.x_min, g.y_min, g.dx, g.n_det, g.s_min, g.ds) == \
        (n0, n1, float(lo[0]), float(lo[1]), dx, n_det, -rho, 2.0 * rho / n_det)
    assert np.array_equal(g.angles, (np.arange(na, dtype=np.float64) + 0.5) * (pi / na))
    assert g.dphi == pi / na
    assert g.range_weight == (pi / na) * g.ds / (g.dx * g.dx)
    assert g.angle_weights is None
    assert np.array_equal(g.range_weights, np.full(na, g.range_weight))


@pytest.mark.parametrize('na,a0,a1', [(60, 0.0, pi / 2), (60, pi / 3, 2 * pi / 3), (7, -pi / 6, pi / 6), (1, 0.0, pi)])
def test_from_angle_range(na, a0, a1):
    g = G.from_angle_range((64, 64), na, a0, a1)
    ref = G.from_im_shape((64, 64), na)
    step = (a1 - a0) / na
    assert np.allclose(g.angles, a0 + (np.arange(na) + 0.5) * step, rtol=0, atol=1e-15)
    assert g.dphi == pytest.approx((a1 - a0) / na, rel=1e-15)
    assert g.angle_weights is None
    assert (g.n_det, g.s_min, g.ds, g.x_min, g.dx) == (ref.n_det, ref.s_min, ref.ds, ref.x_min, ref.dx)
    with pytest.raises(ValueError):
        G.from_angle_range((64, 64), na, a1, a0)
    with pytest.raises(ValueError):
        G.from_angle_range((64, 64), 0, a0, a1)


def test_from_angles_follows_the_odl_rule():
    # sorted views 0, 0.1, 0.3, 0.6: cell edges -0.05 | 0.05 | 0.2 | 0.45 | 0.75 -> cells 0.1, 0.15, 0.25, 0.3,
    # span 0.8, mean cell 0.2
    g = G.from_angles((32, 32), [0.0, 0.1, 0.3, 0.6])
    assert g.dphi == pytest.approx(0.2, rel=1e-14)
    assert np.allclose(g.angle_weights, [0.5, 0.75, 1.25, 1.5], rtol=0, atol=1e-14)
    assert np.allclose(g.range_weights, g.dphi * np.array([0.5, 0.75, 1.25, 1.5]) * g.ds / g.dx ** 2, rtol=1e-14)
    # the caller's order is kept
    p = G.from_angles((32, 32), [0.3, 0.0, 0.6, 0.1])
    assert np.array_equal(p.angles, [0.3, 0.0, 0.6, 0.1])
    assert np.allclose(p.angle_weights, [1.25, 0.5, 1.5, 0.75], rtol=0, atol=1e-14)


@pytest.mark.parametrize('angles', [_golden_angles(37), _golden_angles(180),
                                    np.sort(np.random.default_rng(3).choice(180, 60, replace=False)) * pi / 180 + pi / 360])
def test_from_angles_weights_sum_to_n(angles):
    g = G.from_angles((32, 32), angles)
    assert g.angle_weights is not None and np.all(g.angle_weights > 0)
    assert g.angle_weights.sum() == pytest.approx(g.n_angles, rel=1e-12)
    assert g.dphi * g.n_angles == pytest.approx(g.angle_span, rel=1e-14)


def test_from_angles_uniform_list_has_no_weights():
    ref = G.from_im_shape((48, 48), 30)
    g = G.from_angles((48, 48), ref.angles[::-1])
    assert g.angle_weights is None
    assert g.dphi == pytest.approx(ref.dphi, rel=1e-12)
    assert G.from_angles((48, 48), [0.7]).angle_weights is None


@pytest.mark.parametrize('angles', [[0.1, 0.2, 0.1], [], [0.0, np.nan]])
def test_from_angles_rejects_bad_lists(angles):
    with pytest.raises(ValueError):
        G.from_angles((32, 32), angles)


# ------------------------------------------------------------------------------------------------ oracle ---
@pytest.mark.parametrize('kind', ['golden', 'wedge_random_weights'])
def test_weighted_c_backprojector_equals_weighted_bp_matrix(kind):
    if kind == 'golden':
        geom = W.geometry(G.from_angles((48, 40), _golden_angles(23)))
    else:
        rng = np.random.default_rng(5)
        w = rng.uniform(0.3, 2.0, 17)
        geom = W.geometry(G.from_angle_range((48, 40), 17, 0.2, 1.9))
        geom.w = w / w.mean()
    rng = np.random.default_rng(0)
    y = rng.standard_normal((2, *geom.obs_shape)).astype(np.float32)
    z = W.bp(geom, y)
    z2 = (W.bp_matrix(geom) @ y.reshape(2, -1).T.astype(np.float64)).T.reshape(z.shape)
    assert rel_l2(z, z2) < 1e-6


@pytest.mark.parametrize('case', ['wedge90', 'wedge120', 'golden37', 'random60of180', 'full60'])
def test_adjoint_of_ones_is_the_sum_of_the_cells(case):
    n = 64
    if case == 'wedge90':
        g = G.from_angle_range((n, n), 60, 0.0, pi / 2)
    elif case == 'wedge120':
        g = G.from_angle_range((n, n), 60, 0.0, 2 * pi / 3)
    elif case == 'golden37':
        g = G.from_angles((n, n), _golden_angles(37))
    elif case == 'random60of180':
        keep = np.sort(np.random.default_rng(7).choice(180, 60, replace=False))
        g = G.from_angles((n, n), (keep + 0.5) * pi / 180)
    else:
        g = G.from_im_shape((n, n), 60)
    geom = W.geometry(g)
    z = W.bp(geom, np.ones((1, *geom.obs_shape), np.float32))[0]
    # pixels whose detector coordinate lies inside the detector for every view: the inscribed disc
    x = geom.x_min + (np.arange(n) + 0.5) * geom.dx
    inside = (x[:, None] ** 2 + x[None, :] ** 2) < (0.9 * (-geom.s_min)) ** 2
    total = float(np.sum(g.dphi * g.view_weights))
    assert total == pytest.approx(g.angle_span, rel=1e-12)
    assert np.max(np.abs(z[inside] - total)) < 1e-6 * total
    if case.startswith('wedge'):
        assert total == pytest.approx(pi / 2 if case == 'wedge90' else 2 * pi / 3, rel=1e-12)
    elif case == 'full60':
        assert total == pytest.approx(pi, rel=1e-15)
    else:                                    # a full-range set: its ODL cells cover ~[0, pi)
        assert abs(total - pi) < 2 * pi / g.n_angles


def test_unit_weights_change_nothing():
    base = O.OracleGeometry((40, 56), 11)
    unit = W.geometry(G.from_im_shape((40, 56), 11))
    assert np.array_equal(unit.w, np.ones(11)) and np.array_equal(unit.angles, base.angles) and unit.dphi == base.dphi
    rng = np.random.default_rng(1)
    y = rng.standard_normal((2, *base.obs_shape)).astype(np.float32)
    assert np.array_equal(O.bp(base, y), W.bp(unit, y))
    assert (O.bp_matrix(base) != W.bp_matrix(unit)).nnz == 0
    ref = O.fbp(base, y)
    assert np.max(np.abs(W.fbp(unit, y) - ref)) < 1e-5 * np.max(np.abs(ref))


def test_weighted_fbp_beats_unweighted_on_a_nonuniform_full_range_set():
    n = 128
    g = G.from_angles((n, n), _golden_angles(180))
    weighted = W.geometry(g)
    unweighted = W.geometry(g, weighted=False)
    phantoms = disk_ellipses(3, n, seed=1)
    for k in range(phantoms.shape[0]):
        x = phantoms[k:k + 1, 0]
        y = O.fp(weighted, x.astype(np.float32))
        e_w = rel_l2(W.fbp(weighted, y), x)
        e_u = rel_l2(W.fbp(unweighted, y), x)
        assert e_w < e_u, (k, e_w, e_u)
