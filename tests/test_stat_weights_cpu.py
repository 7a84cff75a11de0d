"""Measurement weights (penalised weighted least squares) without a GPU: the float64 oracle of the weighted system,
the Poisson simulation, the host-side validation of the weights and the plumbing of the factories."""
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch

import angle_set_oracle as AO
import stat_weights_oracle as SW
from fp64_reference import cg64 as cg64_unweighted


def _G():
    from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D
    return ParallelBeamGeometry2D


def _og(shape=(24, 24), na=8):
    return AO.geometry(_G().from_im_shape(shape, na))


def _weights(og, batch, seed=3):
    rng = np.random.default_rng(seed)
    return 10.0 ** rng.uniform(-1.5, 1.5, size=(batch, 1, og.n_angles, og.n_det))


def test_unit_weights_are_the_unweighted_reference():
    og = _og()
    J, Bm = SW.matrices(og)
    rng = np.random.default_rng(0)
    x0, rhs = rng.standard_normal((2, 3, 1, *og.im_shape))
    ones = np.ones((og.n_angles, og.n_det))
    ref = cg64_unweighted(og, x0, rhs, 0.05, 4)
    np.testing.assert_allclose(SW.cg64(J, Bm, og, x0, rhs, 0.05, 4, ones), ref, rtol=0, atol=1e-12 * np.abs(ref).max())


@pytest.mark.parametrize('adjoint', ['pixel', 'matched'])
def test_zero_weight_views_are_deleted_views(adjoint):
    og = _og()
    J, Bm = SW.matrices(og, adjoint)
    drop = [1, 5]
    w = np.ones((og.n_angles, og.n_det))
    w[drop] = 0.0
    keep = np.ones(og.n_angles * og.n_det, dtype=bool)
    for k in drop:
        keep[k * og.n_det:(k + 1) * og.n_det] = False
    Jk, Bk = J[keep], Bm[:, keep]
    rng = np.random.default_rng(1)
    v, rhs = rng.standard_normal((2, 2, 1, *og.im_shape))
    n = og.n0 * og.n1
    ref_op = lambda a: a + 0.05 * (Bk @ (Jk @ a))             # noqa: E731
    vc = v.reshape(-1, n).T
    got = SW.normal64(J, Bm, og, v, 0.05, w)
    np.testing.assert_allclose(got, ref_op(vc).T.reshape(v.shape), rtol=0, atol=1e-12 * np.abs(got).max())
    # the CG iterates of the two systems: the reduced matrices, unweighted
    x = SW.cg_cols(ref_op, vc.copy(), rhs.reshape(-1, n).T, 4)
    got = SW.cg64(J, Bm, og, v, rhs, 0.05, 4, w)
    np.testing.assert_allclose(got, x.T.reshape(v.shape), rtol=0, atol=1e-12 * np.abs(got).max())


def test_matched_weighted_operator_is_symmetric():
    geom = _G().from_angles((24, 24), np.sort(np.random.default_rng(4).uniform(0, np.pi, 9)))
    og = AO.geometry(geom)
    J, Bm = SW.matrices(og, 'matched')
    w = _weights(og, 1)[0, 0]
    rng = np.random.default_rng(5)
    u, v = rng.standard_normal((2, 1, 1, *og.im_shape))
    lhs = float((u * SW.normal64(J, Bm, og, v, 0.1, w)).sum())
    rhs = float((SW.normal64(J, Bm, og, u, 0.1, w) * v).sum())
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), 1.0), (lhs, rhs)


class _CpuTrafo:
    """A CPU stand-in of the ray transform: the oracle's Joseph matrix for A, its transpose for A*."""

    def __init__(self, og):
        self.og, self.im_shape, self.obs_shape = og, og.im_shape, og.obs_shape
        self.J = AO.matrices(og)[0]
        self.Bm = AO.matrices(og)[1]

    def __call__(self, x):
        a = x.detach().double().reshape(-1, self.og.n0 * self.og.n1).numpy().T
        return torch.from_numpy((self.J @ a).T.reshape(*x.shape[:-2], *self.obs_shape)).float()

    trafo = __call__

    def trafo_adjoint(self, y):
        a = y.detach().double().reshape(-1, self.og.n_angles * self.og.n_det).numpy().T
        return torch.from_numpy((self.Bm @ a).T.reshape(*y.shape[:-2], *self.im_shape)).float()


def test_simulate_poisson_matches_numpy():
    from diffusion_models_dev_project_b200 import simulate_poisson
    og = _og((32, 32), 12)
    rt = _CpuTrafo(og)
    x = torch.rand(3, 1, 32, 32, generator=torch.Generator().manual_seed(2))
    photons, mu = 2e3, 0.05
    y, w = simulate_poisson(x, rt, photons, mu, np.random.default_rng(9))
    counts, y_ref, w_ref = SW.poisson64(rt(x).numpy(), photons, mu, np.random.default_rng(9))
    assert y.dtype == w.dtype == torch.float32 and y.shape == w.shape == (3, 1, 12, og.n_det)
    # the counts are recovered from y exactly: same generator, same draws
    np.testing.assert_array_equal(np.rint(photons * np.exp(-mu * y.double().numpy())).clip(min=0.1),
                                  np.where(counts < 1, 0.1, counts))
    np.testing.assert_allclose(y.numpy(), y_ref, rtol=1e-7, atol=1e-7 * np.abs(y_ref).max())
    np.testing.assert_allclose(w.numpy(), w_ref, rtol=1e-7, atol=0)
    np.testing.assert_allclose(w.double().mean(dim=(1, 2, 3)).numpy(), 1.0, rtol=1e-6)


def _rt():
    from diffusion_models_dev_project_b200 import B200RayTrafo
    return B200RayTrafo((24, 24), 8)


@pytest.mark.parametrize('case', ['shape', 'rank5', 'dtype', 'nan', 'inf', 'negative', 'cpu', 'not_a_tensor'])
def test_weights_are_validated_on_creation(case):
    from diffusion_models_dev_project_b200 import MeasurementWeights
    rt = _rt()
    obs = rt.obs_shape
    w = {'shape': torch.ones(obs[0], obs[1] + 1), 'rank5': torch.ones(2, 1, 3, *obs),
         'dtype': torch.ones(*obs, dtype=torch.float64), 'nan': torch.ones(*obs), 'inf': torch.ones(*obs),
         'negative': torch.ones(*obs), 'cpu': torch.ones(1, 1, *obs), 'not_a_tensor': np.ones(obs, np.float32)}[case]
    if case == 'nan':
        w[2, 3] = float('nan')
    if case == 'inf':
        w[0, 0] = float('inf')
    if case == 'negative':
        w[1, 1] = -1e-3
    err = TypeError if case in ('dtype', 'not_a_tensor') else ValueError
    with pytest.raises(err):
        MeasurementWeights(rt, w)


def test_sharded_operator_rejects_weights():
    from diffusion_models_dev_project_b200 import MeasurementWeights, NormalOp
    from diffusion_models_dev_project_b200.sharding import AngleShardedRayTrafo
    sh = AngleShardedRayTrafo(_rt())
    w = torch.ones(*sh.obs_shape)
    with pytest.raises(ValueError, match='measurement weights'):
        sh.normal_op(0.1, weights=w)
    with pytest.raises(ValueError, match='measurement weights'):
        sh.normal_apply(torch.zeros(1, 1, 24, 24), 0.1, weights=w)
    with pytest.raises(TypeError, match='sharded'):
        MeasurementWeights(sh, w)
    with pytest.raises(TypeError, match='sharded'):
        NormalOp(sh, 0.1, weights=w)


def _args(**kw):
    base = dict(method='dds', num_steps=4, pct_chain_elapsed=0, eta=0.15, gamma=0.02, cg_iter=3, penalty=1.0,
                early_stopping_pct=1.0, adaptation='full', num_optim_step=1, adapt_freq=1, lr=1e-3, tv_penalty=1e-4,
                add_cg=True, dc_type='cg', lora_include_blocks=None, lora_rank=4)
    base.update(kw)
    return NS(**base)


def _config():
    return NS(device='cpu', sampling=NS(batch_size=2, eps=1e-3, travel_length=1, travel_repeat=1),
              model=NS(in_channels=1))


def test_factories_bind_weighted_rhs_and_pass_the_weights():
    import diffusion_models_dev_project_b200 as pkg
    og = _og()
    rt = _CpuTrafo(og)
    y = torch.rand(2, 1, *og.obs_shape, generator=torch.Generator().manual_seed(1))
    w = torch.from_numpy(_weights(og, 2)).float()
    sde = pkg.DDPM()
    score = torch.nn.Conv2d(1, 1, 1)
    sampler = pkg.get_standard_sampler(_args(), _config(), score, sde, rt, observation=y, weights=w)
    kw = sampler.predictor.keywords
    assert kw['cg_kwargs'] == {'max_iter': 3, 'weights': w}
    assert torch.equal(kw['rhs'], rt.trafo_adjoint(w * y))
    sampler = pkg.get_standard_sampler(_args(), _config(), score, sde, rt, observation=y)
    assert sampler.predictor.keywords['cg_kwargs'] == {'max_iter': 3}
    assert torch.equal(sampler.predictor.keywords['rhs'], rt.trafo_adjoint(y))
    with pytest.raises(ValueError, match='dds'):
        pkg.get_standard_sampler(_args(method='dps'), _config(), score, sde, rt, observation=y, weights=w)
    sampler = pkg.get_standard_adapted_sampler(_args(), _config(), score, sde, rt, observation=y, weights=w)
    kw = sampler.predictor.keywords
    assert kw['cg_kwargs']['weights'] is w and torch.equal(kw['rhs'], rt.trafo_adjoint(w * y))
    loss_fn = kw['adapt_fn'].keywords['loss_fn']
    assert loss_fn.weights is w
    x = torch.rand(2, 1, *og.im_shape)
    expect = torch.mean(w * (rt(x) - y).pow(2)) + 1e-4 * pkg.tv_loss(x)
    assert torch.allclose(loss_fn(x=x), expect, rtol=1e-6)


def test_predictor_tensor_path_solves_the_weighted_system():
    """A non-B200 operator keeps the tensor path: the predictor's CG runs on ``v + gamma A*(W A v)``, and the
    predictor takes W from its solver options."""
    import diffusion_models_dev_project_b200 as pkg
    from diffusion_models_dev_project_b200.samplers.utils import _make_op
    og = _og()
    rt = _CpuTrafo(og)
    w = torch.from_numpy(_weights(og, 2)).float()
    v = torch.rand(2, 1, *og.im_shape, generator=torch.Generator().manual_seed(4))
    J, Bm = SW.matrices(og)
    got = _make_op(rt, 0.05, w)(v)
    ref = SW.normal64(J, Bm, og, v.numpy(), 0.05, w.numpy())
    np.testing.assert_allclose(got.numpy(), ref, rtol=1e-5, atol=1e-5 * np.abs(ref).max())
    sde = pkg.DDPM()
    score = lambda x, t: torch.zeros_like(x)                                  # noqa: E731
    t = (torch.full((2,), 500.), torch.full((2,), 490.))
    rhs = rt.trafo_adjoint(w * rt(v))
    torch.manual_seed(0)
    _, xhat0 = pkg.decomposed_diffusion_sampling_sde_predictor(
        score, sde, v, rhs, t, 0.0, 0.05, 1.0, {'max_iter': 3, 'weights': w}, ray_trafo=rt)
    xa = pkg.cg(op=_make_op(rt, 0.05, w), x=xhat0, rhs=xhat0 + 0.05 * rhs, n_iter=3)
    xb = pkg.cg(op=_make_op(rt, 0.05), x=xhat0, rhs=xhat0 + 0.05 * rhs, n_iter=3)
    torch.manual_seed(0)
    x_next, _ = pkg.decomposed_diffusion_sampling_sde_predictor(
        score, sde, v, rhs, t, 0.0, 0.05, 1.0, {'max_iter': 3, 'weights': w}, ray_trafo=rt)
    expect = pkg.ddim(sde=sde, s=torch.zeros_like(v), xhat=xa, time_step=t, step_size=1.0, eta=0.0,
                      use_simplified_eqn=False)
    assert torch.allclose(x_next, expect, rtol=1e-5, atol=1e-6) and not torch.allclose(xa, xb, rtol=1e-3)
