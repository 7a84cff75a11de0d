"""CPU tests of the host-side mirror of the reference interfaces and of the C-ABI library
(loads, exports every declared symbol, rejects use without a GPU -- no compute calls here)."""
import functools
import json
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, rel_l2
from oracle import oracle as O

import diffusion_models_dev_project_b200 as pkg
from diffusion_models_dev_project_b200 import _lib


# ------------------------------------------------------------------ C ABI ----
def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'scd_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(scd_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), 'libscd_b200.so does not export %s' % n
        assert n in _lib.SIGNATURES, 'python binding missing for %s' % n
    assert set(_lib.SIGNATURES) == set(names)
    assert b'sm_100a' in lib.scd_version()


def test_library_contains_sm100a_code_with_bulk_copies():
    import shutil
    import subprocess
    if shutil.which('cuobjdump') is None:
        pytest.skip('cuobjdump not available')
    out = subprocess.run(['cuobjdump', '-lelf', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'sm_100a' in out
    sass = subprocess.run(['cuobjdump', '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'UBLKCP' in sass          # cp.async.bulk (TMA unit): packed strips / sinogram segments
    assert 'UTMALDG' in sass         # cp.async.bulk.tensor: strips gathered from the interleaved image
    assert 'SYNCS' in sass           # mbarrier


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour without a GPU')
def test_no_cpu_fallback():
    rt = pkg.B200RayTrafo((32, 32), 6)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        rt(torch.rand(1, 1, 32, 32))
    with pytest.raises(RuntimeError):
        rt.trafo_adjoint(torch.rand(1, 1, *rt.obs_shape))
    import ctypes as C
    lib = _lib.load()
    ang = np.array([0.1, 0.2])
    desc = _lib.GeomDesc(n0=8, n1=8, x_min=-4, y_min=-4, dx=1, n_angles=2,
                         angles=ang.ctypes.data_as(C.POINTER(C.c_double)), n_det=13, s_min=-6, ds=1, adj_scale=1)
    h = C.c_void_p()
    assert lib.scd_geom_create(C.byref(desc), C.byref(h)) == _lib.SCD_E_NODEVICE
    assert 'no CPU path' in _lib.last_error() or 'CUDA' in _lib.last_error()


def test_geom_create_rejects_bad_arguments():
    import ctypes as C
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.scd_geom_create(None, C.byref(h)) == _lib.SCD_E_INVALID
    desc = _lib.GeomDesc(n0=0, n1=8)
    assert lib.scd_geom_create(C.byref(desc), C.byref(h)) == _lib.SCD_E_INVALID
    assert 'invalid geometry' in _lib.last_error()
    assert lib.scd_geom_destroy(None) == 0


# ---------------------------------------------------------------- geometry ----
def test_geometry_object():
    g = pkg.ParallelBeamGeometry2D.from_im_shape((256, 256), 60)
    o = O.OracleGeometry((256, 256), 60)
    assert (g.n_det, g.x_min, g.s_min, g.ds) == (o.n_det, o.x_min, o.s_min, o.ds)
    assert np.array_equal(g.angles, o.angles)
    rt = pkg.B200RayTrafo((501, 501), 1200)
    assert rt.obs_shape == (1200, 711) and rt.im_shape == (501, 501)
    assert not hasattr(rt, 'resize')
    assert isinstance(rt, pkg.BaseRayTrafo) and isinstance(rt, torch.nn.Module)
    assert rt.to('cpu') is rt
    with pytest.raises(NotImplementedError):
        pkg.B200RayTrafo((64, 64), 10, impl='something')
    assert pkg.SimpleTrafo is pkg.B200RayTrafo


class _CpuTrafo(pkg.BaseRayTrafo):
    """BaseRayTrafo subclass over the oracle matrices: exercises the adapters of the boundary type."""

    def __init__(self, geom, odl_autograd=False):
        super().__init__(geom.im_shape, geom.obs_shape)
        self.rt = O.OracleRayTrafo(geom, odl_autograd=odl_autograd)

    def trafo(self, x):
        return self.rt.trafo(x)

    def trafo_adjoint(self, y):
        return self.rt.trafo_adjoint(y)

    trafo_flat = pkg.BaseRayTrafo._trafo_flat_via_trafo
    trafo_adjoint_flat = pkg.BaseRayTrafo._trafo_adjoint_flat_via_trafo_adjoint


def test_base_ray_trafo_adapters():
    geom = O.OracleGeometry((16, 16), 5)
    rt = _CpuTrafo(geom)
    x = torch.rand(2, 3, 16, 16)
    y = rt(x)
    assert y.shape == (2, 3, 5, geom.n_det)
    yf = rt.trafo_flat(x.reshape(6, -1).T)
    assert yf.shape == (5 * geom.n_det, 6) and torch.equal(yf.T.reshape(y.shape), y)
    xf = rt.trafo_adjoint_flat(yf)
    assert torch.allclose(xf.T.reshape(x.shape), rt.trafo_adjoint(y))
    with pytest.raises(NotImplementedError):
        rt.fbp(y)


# ------------------------------------------------------- schedule / DDPM -----
def test_schedule_and_ddpm_match_reference_golden():
    with open(os.path.join(GOLDEN, 'schedule.json')) as f:
        ref = json.load(f)
    for key, val in ref['jump'].items():
        assert pkg._schedule_jump(*[int(v) for v in key.split(',')]) == val
    sde = pkg.DDPM()
    for n, pairs in ref['pairs'].items():
        kw = {'num_steps': int(n), 'travel_length': 1, 'travel_repeat': 1}
        s = pkg.BaseSampler(score=None, sde=sde, predictor=None, sample_kwargs=kw)
        _, steps = s._schedule()
        assert [list(p) for p in steps] == pairs
    t = torch.tensor(ref['abar']['t'])
    assert sde._compute_alpha_cumprod(t).numpy().view(np.uint32).tolist() == ref['abar']['bits']
    assert sde.marginal_prob_mean(t).numpy().view(np.uint32).tolist() == ref['mean']
    assert sde.marginal_prob_std(t).numpy().view(np.uint32).tolist() == ref['std']
    assert np.array_equal(sde.alpha_bar_table().numpy(), np.load(os.path.join(GOLDEN, 'abar_table.npy')))
    assert sde.prior_sampling([2, 1, 4, 4]).shape == (2, 1, 4, 4)
    kw = {'num_steps': 100, 'travel_length': 1, 'travel_repeat': 1, 'early_stopping_pct': 0.5}
    _, steps = pkg.BaseSampler(None, sde, None, kw)._schedule()
    assert len(steps) == 50


def test_ve_vp_schedules():
    t = torch.tensor([0.1, 0.5, 1.0])
    ve, vp = pkg.VESDE(0.01, 100), pkg.VPSDE(0.1, 10)
    assert torch.allclose(ve.marginal_prob_std(t), 0.01 * (100 / 0.01) ** t)
    assert torch.equal(ve.marginal_prob_mean(t), torch.ones(3))
    lm = -0.25 * t ** 2 * 9.9 - 0.5 * t * 0.1
    assert torch.allclose(vp.marginal_prob_mean(t), torch.exp(lm))
    assert torch.allclose(vp.marginal_prob_std(t), torch.sqrt(1 - torch.exp(2 * lm)))
    assert pkg._SCORE_PRED_CLASSES == [pkg.VPSDE, pkg.VESDE] and pkg._EPSILON_PRED_CLASSES == [pkg.DDPM]


# ------------------------------------- generic (tensor-op) paths vs reference --
def test_tweedie_and_ddim_tensor_paths_match_reference_golden(golden, monkeypatch):
    """On CPU tensors apTweedy / ddim run as tensor ops (the path autograd uses): bit-exact vs reference."""
    d = golden('tweedie_ddim.npz')
    sde = pkg.DDPM()
    x, s, xhat = (torch.from_numpy(d[k]) for k in ('x', 's', 'xhat'))
    for ci, (t, tp) in enumerate(d['cases']):
        tt, tpv = torch.ones(3) * float(t), torch.ones(3) * float(tp)
        assert np.array_equal(pkg.apTweedy(s=s, x=x, sde=sde, time_step=tt).numpy(), d['tweedie_%d' % ci])
        for eta in (0.0, 0.15, 0.85):
            torch.manual_seed(77 + ci)
            out = pkg.ddim(sde=sde, s=s, xhat=xhat, time_step=(tt, tpv), step_size=1, eta=eta,
                           use_simplified_eqn=True)
            assert np.array_equal(out.numpy(), d['ddim_%d_%g' % (ci, eta)])


def test_cg_tensor_path_matches_reference_golden(golden):
    d = golden('cg_small.npz')
    rt = O.OracleRayTrafo(O.OracleGeometry((32, 32), 12))
    x0, rhs = torch.from_numpy(d['x0']), torch.from_numpy(d['rhs'])
    for gamma in (0.01, 1.0):
        op = lambda v: v + gamma * rt.trafo_adjoint(rt(v))      # noqa: E731
        for k in (0, 1, 2, 5):
            out = pkg.cg(op=op, x=x0, rhs=rhs, n_iter=k).numpy()
            # (p*d).sum vs norm()**2: same maths, different reduction -> round-off only
            assert rel_l2(out, d['x_g%g_k%d' % (gamma, k)]) < (1e-6 if gamma < 1 else 5e-4)


def test_sampler_with_generic_operator_matches_reference_chain(golden):
    """BaseSampler + DDS predictor of this package, driven on CPU with the oracle operator,
    reproduces the reference sampler's reconstruction (same seeds)."""
    from scorenet import BlurScore
    d = golden('dds_small.npz')
    rt = O.OracleRayTrafo(O.OracleGeometry((64, 64), 16))
    sde, score = pkg.DDPM(), BlurScore()
    y = torch.from_numpy(d['y'])
    kw = {'num_steps': 10, 'batch_size': 2, 'start_time_step': 0, 'im_shape': [1, 64, 64], 'eps': 1e-3,
          'travel_length': 1, 'travel_repeat': 1,
          'predictor': {'eta': 0.15, 'gamma': 0.05, 'use_simplified_eqn': True, 'ray_trafo': rt}}
    predictor = functools.partial(pkg.decomposed_diffusion_sampling_sde_predictor, score=score, sde=sde,
                                  rhs=rt.trafo_adjoint(y), cg_kwargs={'max_iter': 3})
    sampler = pkg.BaseSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=kw, device='cpu')
    torch.manual_seed(11)
    recon = sampler.sample(logging=False)
    assert rel_l2(recon.numpy(), d['recon']) < 1e-5


def test_adaptation_loss_tensor_expression_and_tv():
    """adaptation_loss on a non-B200 operator evaluates the reference's expression (src/utils/exp_utils.py:256-257);
    tv_loss matches a direct restatement of src/samplers/adaptation.py:7-11."""
    rt = O.OracleRayTrafo(O.OracleGeometry((16, 16), 6))
    g = torch.Generator().manual_seed(2)
    x = torch.rand(2, 1, 16, 16, generator=g, requires_grad=True)
    y = rt(torch.rand(1, 1, 16, 16, generator=g))
    loss = pkg.adaptation_loss(x, y, rt, 1e-2)
    ref = torch.mean((rt(x) - y).pow(2)) + 1e-2 * pkg.tv_loss(x)
    assert torch.equal(loss, ref)
    loss.backward()
    assert torch.isfinite(x.grad).all() and float(x.grad.abs().max()) > 0
    xn = x.detach().numpy()
    dh = np.abs(xn[..., :, 1:] - xn[..., :, :-1])[..., :-1, :]
    dw = np.abs(xn[..., 1:, :] - xn[..., :-1, :])[..., :, :-1]
    assert abs(float(pkg.tv_loss(x)) - float((dh + dw).sum())) < 1e-4


def test_metrics_psnr_ssim():
    rng = np.random.default_rng(0)
    gt = rng.random((64, 48))
    assert pkg.PSNR(gt, gt) == float('inf') and abs(pkg.SSIM(gt, gt) - 1.0) < 1e-12
    noisy = gt + 0.1 * rng.standard_normal(gt.shape)
    mse = np.mean((noisy - gt) ** 2)
    assert abs(pkg.PSNR(noisy, gt) - 10 * np.log10((gt.max() - gt.min()) ** 2 / mse)) < 1e-9
    s1, s2 = pkg.SSIM(noisy, gt), pkg.SSIM(gt + 0.3 * rng.standard_normal(gt.shape), gt)
    assert 0 < s2 < s1 < 1                                   # monotone in the noise level
    assert abs(pkg.SSIM(gt + 0.2, gt, data_range=1.0) - pkg.SSIM(gt, gt + 0.2, data_range=1.0)) < 1e-12   # symmetric


def test_other_guidance_predictors_match_reference(golden):
    """Euler-Maruyama (plain / naive / DPS), Langevin corrector and ancestral sampling (plain / DPS): one
    step each on CPU with the oracle operator against the reference's own functions (same seeds)."""
    from scorenet import BlurScore
    d = golden('predictors_small.npz')
    rt = O.OracleRayTrafo(O.OracleGeometry((24, 24), 8))
    x = torch.from_numpy(d['x'])
    y = torch.from_numpy(d['y'])
    nll = lambda v: torch.linalg.norm(y - rt(v))          # noqa: E731

    class VpScore(torch.nn.Module):
        def forward(self, v, t):
            return -0.7 * v + 0.1 * torch.tanh(v) * t[:, None, None, None]
    vp, vscore = pkg.VPSDE(), VpScore()
    tv = torch.ones(2) * 0.4
    for name, kw in (('em_plain', {}), ('em_naive', dict(nloglik=nll, datafitscale=0.4, penalty=0.3, aTweedy=False)),
                     ('em_dps', dict(nloglik=nll, datafitscale=0.4, penalty=0.3, aTweedy=True))):
        torch.manual_seed(5)
        a, b = pkg.Euler_Maruyama_sde_predictor(score=vscore, sde=vp, x=x.clone(), time_step=tv, step_size=1e-2, **kw)
        assert rel_l2(a.numpy(), d[name + '_x']) < 1e-6 and rel_l2(b.numpy(), d[name + '_mean']) < 1e-6, name
    torch.manual_seed(6)
    out = pkg.Langevin_sde_corrector(score=vscore, sde=vp, x=x.clone(), time_step=tv, nloglik=nll, datafitscale=0.4,
                                     penalty=0.3, corrector_steps=2)
    assert rel_l2(out.numpy(), d['langevin']) < 1e-6
    sde, score = pkg.DDPM(), BlurScore()
    ts = (torch.ones(2) * 400., torch.ones(2) * 390.)
    for name, kw in (('anc_plain', {}), ('anc_dps', dict(nloglik=nll, penalty=0.5))):
        torch.manual_seed(7)
        a, b = pkg.Ancestral_Sampling(score=score, sde=sde, x=x.clone(), time_step=ts, step_size=1, **kw)
        assert rel_l2(a.numpy(), d[name + '_x']) < 1e-6 and rel_l2(b.numpy(), d[name + '_xhat0']) < 1e-6, name


def test_adapted_predictor_and_adapt_run_with_autograd():
    """SCD step on CPU with a tiny trainable score: _adapt changes the trainable parameters through
    Tweedie -> CG -> loss, and the adapted predictor returns finite tensors of the right shape."""
    geom = O.OracleGeometry((16, 16), 6)
    rt = O.OracleRayTrafo(geom)

    class LoraInjectedConv2d(torch.nn.Module):          # class name is what _has_lora() looks for
        def __init__(self):
            super().__init__()
            self.conv = torch.nn.Conv2d(1, 1, 3, padding=1)
            self.scale = 1.0

        def forward(self, x):
            return self.conv(x) * self.scale

    class Score(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l = LoraInjectedConv2d()

        def forward(self, x, t):
            return 0.1 * x + self.l(x)

    torch.manual_seed(0)
    score, sde = Score(), pkg.DDPM()
    gt = torch.rand(1, 1, 16, 16)
    y = rt(gt)
    rhs = rt.trafo_adjoint(y)
    loss_fn = lambda x: torch.mean((rt(x) - y).pow(2)) + 1e-6 * pkg.tv_loss(x)   # noqa: E731
    before = score.l.conv.weight.detach().clone()
    x = torch.randn(1, 1, 16, 16)
    t = torch.ones(1) * 500.
    pkg._adapt(x=x, score=score, sde=sde, ray_trafo=rt, loss_fn=loss_fn, time_step=t, rhs=rhs, num_steps=2,
               lr=1e-2, gamma=0.1, n_iter=1)
    assert not torch.equal(before, score.l.conv.weight.detach())
    adapt_fn = functools.partial(pkg._adapt, score=score, sde=sde, loss_fn=loss_fn, num_steps=1, lr=1e-3)
    for dc in ('cg', 'gd', 'none'):
        xn, x0 = pkg.adapted_ddim_sde_predictor(
            score=score, sde=sde, x=x, time_step=(t, torch.ones(1) * 490.), eta=0.85, step_size=1,
            adapt_fn=adapt_fn, use_adapt=True, ray_trafo=rt, add_cg=True, dc_type=dc, gamma=0.1,
            cg_kwargs={'max_iter': 1}, rhs=rhs)
        assert xn.shape == x.shape and torch.isfinite(xn).all() and torch.isfinite(x0).all()
    assert score.l.scale == 1.0
    assert float(pkg.tv_loss(torch.ones(1, 1, 4, 4))) == 0.0


def test_adapted_sampling_matches_reference_chain(golden):
    """BASELINE config 5 (SCD adapted sampling) on a CPU-sized chain: this package's factory, `_adapt`,
    adapted predictor and sampler against the outputs of the reference's own
    get_standard_adapted_sampler / _adapt / adapted_ddim_sde_predictor / BaseSampler
    (tests/golden/make_golden.py:adapted_fixture) -- reconstruction and the adapted parameters."""
    from make_golden_args import adapted_args, adapted_config
    from scorenet import AdaptableScore
    from diffusion_models_dev_project_b200.utils import exp_utils as E
    d = golden('adapted_small.npz')
    geom = O.OracleGeometry(tuple(int(v) for v in d['im']), int(d['num_angles']))
    rt = _CpuTrafo(geom, odl_autograd=True)
    y = torch.from_numpy(d['y'])
    for dc in ('cg', 'gd'):
        score = AdaptableScore(r=2, seed=0)
        sampler = E.get_standard_adapted_sampler(adapted_args(dc), adapted_config(2, 'cpu'), score, pkg.DDPM(), rt,
                                                 observation=y, device='cpu')
        torch.manual_seed(13)
        recon = sampler.sample(logging=False)
        assert rel_l2(recon.numpy(), d['recon_' + dc]) < 1e-5, dc
        for name, prm in score.named_parameters():
            assert np.allclose(prm.detach().numpy(), d['param_%s_%s' % (dc, name)], atol=2e-6), (dc, name)
        assert score.adapter.scale == 1.0


def test_cg_hand_written_backward_equals_autograd_through_the_recurrences():
    """The reverse sweep of `_CgSelfAdjointFn` (used for `op = I + gamma A*A` on the CUDA operator, whose
    gradient is `op` itself) against autograd through the tensor recurrences, in float64 on a symmetric
    operator built from the oracle's Joseph matrix."""
    import importlib
    C = importlib.import_module('diffusion_models_dev_project_b200.utils.cg')
    geom = O.OracleGeometry((16, 16), 6)
    J = O.OracleRayTrafo(geom, matched_adjoint=True).matrix.to_dense().double()
    M = torch.eye(256, dtype=torch.float64) + 0.3 * geom.dphi * geom.ds * (J.T @ J)

    def op(v):
        return (v.reshape(v.shape[0], -1) @ M.T).reshape(v.shape)
    gen = torch.Generator().manual_seed(0)
    for k in (0, 1, 3, 5):
        x = torch.randn(2, 1, 16, 16, dtype=torch.float64, generator=gen, requires_grad=True)
        b = torch.randn(2, 1, 16, 16, dtype=torch.float64, generator=gen, requires_grad=True)
        w = torch.randn(2, 1, 16, 16, dtype=torch.float64, generator=gen)
        ref = pkg.cg(op, x, b, k)                                  # generic callable: tensor recurrences + autograd
        gx_ref, gb_ref = torch.autograd.grad((ref * w).sum(), (x, b), allow_unused=True)
        gb_ref = torch.zeros_like(b) if gb_ref is None else gb_ref
        out = C._CgSelfAdjointFn.apply(x, b, lambda v: op(v).detach(), k)
        gx, gb = torch.autograd.grad((out * w).sum(), (x, b))
        assert torch.equal(out, ref)
        assert float((gx - gx_ref).norm() / gx_ref.norm()) < 1e-12, k
        assert float((gb - gb_ref).norm()) <= 1e-12 * max(1.0, float(gb_ref.norm())), k


def test_factories_keep_reference_signatures():
    import inspect
    from diffusion_models_dev_project_b200.utils import exp_utils as E
    assert list(inspect.signature(E.get_standard_sampler).parameters)[:8] == [
        'args', 'config', 'score', 'sde', 'ray_trafo', 'observation', 'filtbackproj', 'device']
    assert list(inspect.signature(E.get_standard_adapted_sampler).parameters)[:8] == [
        'args', 'config', 'score', 'sde', 'ray_trafo', 'observation', 'device', 'complex_y']
    assert list(inspect.signature(pkg.cg).parameters) == ['op', 'x', 'rhs', 'n_iter', 'tol']
    assert list(inspect.signature(pkg.ddim).parameters) == [
        'sde', 's', 'xhat', 'time_step', 'step_size', 'eta', 'use_simplified_eqn']
    assert list(inspect.signature(pkg.decomposed_diffusion_sampling_sde_predictor).parameters) == [
        'score', 'sde', 'x', 'rhs', 'time_step', 'eta', 'gamma', 'step_size', 'cg_kwargs', 'datafitscale',
        'use_simplified_eqn', 'ray_trafo']
    assert list(inspect.signature(pkg.adapted_ddim_sde_predictor).parameters) == [
        'score', 'sde', 'x', 'time_step', 'eta', 'step_size', 'adapt_fn', 'use_adapt', 'datafitscale',
        'use_simplified_eqn', 'ray_trafo', 'add_cg', 'dc_type', 'gamma', 'cg_kwargs', 'rhs']

    class NS(dict):
        __getattr__ = dict.__getitem__
    cfg = NS(sde=NS(type='ddpm', beta_min=1e-4, beta_max=0.02, num_steps=1000),
             data=NS(im_size=64), forward_op=NS(trafo_name='simple_trafo', num_angles=12, impl='odl'))
    assert isinstance(E.get_standard_sde(cfg), pkg.DDPM)
    rt = E.get_standard_ray_trafo(cfg)
    assert isinstance(rt, pkg.B200RayTrafo) and rt.obs_shape[0] == 12


def test_psnr():
    gt = np.zeros((4, 4)); gt[0, 0] = 1.0
    assert pkg.PSNR(gt, gt) == float('inf')
    assert abs(pkg.PSNR(gt + 0.1, gt) - 20.0) < 1e-9


# ------------------------------------------- simulate / data helpers / phantoms / fbp recipe ----
class _MatrixTrafo:
    """Generic CPU operator (dense matrices) with the attributes the data helpers touch."""

    def __init__(self, im_shape=(6, 5), obs_shape=(4, 7), seed=0):
        g = torch.Generator().manual_seed(seed)
        self.im_shape, self.obs_shape = im_shape, obs_shape
        self.M = torch.randn(obs_shape[0] * obs_shape[1], im_shape[0] * im_shape[1], generator=g)

    def trafo(self, x):
        return (x.reshape(*x.shape[:-2], -1) @ self.M.T).reshape(*x.shape[:-2], *self.obs_shape)

    __call__ = trafo

    def fbp(self, y):
        return (y.reshape(*y.shape[:-2], -1) @ self.M).reshape(*y.shape[:-2], *self.im_shape) * 0.01


def test_simulate_reproduces_the_reference_measurements(golden):
    """`simulate` (reference src/physics/simulation.py:12-23) against the `y_i` the REFERENCE's simulate
    produced for the config-1 fixture (tests/golden/make_golden.py: oracle operator, default_rng(1 + i)): same
    random stream, same noise level, no host read-back of the level."""
    d = golden('dds_256.npz')
    ort = O.OracleRayTrafo(O.OracleGeometry((256, 256), 60))
    for i in range(2):
        gt = torch.from_numpy(d['gt_%d' % i])
        y = pkg.simulate(gt, ort, 0.01, rng=np.random.default_rng(1 + i))
        assert y.dtype == torch.float32 and tuple(y.shape) == (1, 1, 60, 365)
        assert np.array_equal(y.numpy(), d['y_%d' % i]), float(np.abs(y.numpy() - d['y_%d' % i]).max())
    y2, level = pkg.simulate(gt, ort, 0.01, rng=np.random.default_rng(2), return_noise_level=True)
    assert np.array_equal(y2.numpy(), d['y_1'])
    assert abs(level - 0.01 * float(ort(gt).abs().mean())) < 1e-12


def test_simulated_dataset_and_get_data_from_ground_truth():
    rt = _MatrixTrafo()
    g = torch.Generator().manual_seed(5)
    imgs = [torch.rand(1, 6, 5, generator=g) for _ in range(4)]
    ds = pkg.SimulatedDataset(imgs, rt, 0.1, use_fixed_seeds_starting_from=3)
    assert len(ds) == 4
    y2, x2, f2 = ds[2]
    assert tuple(y2.shape) == (1, 4, 7) and tuple(x2.shape) == (1, 6, 5) and tuple(f2.shape) == (1, 6, 5)
    ref = pkg.simulate(imgs[2][None], rt, 0.1, rng=np.random.default_rng(3 + 2))[0]
    assert torch.equal(y2, ref) and torch.equal(f2, rt.fbp(ref[None])[0]) and torch.equal(x2, imgs[2])
    assert all(torch.equal(a[0], b[0]) for a, b in zip(ds, [ds[i] for i in range(4)]))      # __iter__ == __getitem__
    with pytest.raises(AssertionError):
        pkg.SimulatedDataset(imgs, rt, 0.1, rng=np.random.default_rng(0))
    shared = pkg.SimulatedDataset(imgs, rt, 0.1, use_fixed_seeds_starting_from=None, rng=np.random.default_rng(0))
    assert not torch.equal(shared[0][0], shared[0][0])             # one generator: consecutive draws differ
    # get_data_from_ground_truth (reference src/utils/exp_utils.py:322-332): 3-D input gains a batch axis
    gt, obs, fbp = pkg.get_data_from_ground_truth(imgs[0], rt, 0.0)
    assert tuple(gt.shape) == (1, 1, 6, 5) and tuple(obs.shape) == (1, 1, 4, 7) and tuple(fbp.shape) == (1, 1, 6, 5)
    assert torch.equal(obs, rt(gt)) and torch.equal(fbp, rt.fbp(obs))
    gt4, _, _ = pkg.get_data_from_ground_truth(gt, rt, 0.0)
    assert gt4 is gt


def test_disk_ellipse_phantoms_are_deterministic_and_normalised():
    """Synthetic stand-in of DiskDistributedEllipsesDataset (reference src/dataset/ellipses.py:121-136 random
    parameters, :72-79 foreground normalisation)."""
    from bench_support.phantoms import disk_ellipses
    a = disk_ellipses(3, 64, seed=1)
    b = disk_ellipses(3, 64, seed=1)
    c = disk_ellipses(3, 64, seed=2)
    assert a.shape == (3, 1, 64, 64) and a.dtype == np.float32
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    assert np.array_equal(disk_ellipses(2, 64, seed=1), a[:2])            # a prefix of the same stream
    for img in a[:, 0]:
        assert img.min() >= 0.0 and abs(img.max() - 1.0) < 1e-6
        r = np.hypot(*np.meshgrid((np.arange(64) + .5) / 32 - 1, (np.arange(64) + .5) / 32 - 1, indexing='ij'))
        assert (img != 0).mean() > 0.05 and img[r > 0.95].max() < 0.5     # mass sits in the central disk


def test_oracle_fbp_recipe():
    """oracle.filter_sinogram restates the reference's zero-padded FFT recipe (src/physics/utils.py:11-33); it
    equals the linear convolution with the Kak-Slaney ramp (what scd_ramp_filter evaluates), and
    fbp(A x) ~ x."""
    geom = O.OracleGeometry((64, 64), 90)
    rng = np.random.default_rng(0)
    y = rng.standard_normal((2, 90, geom.n_det))
    q = O.filter_sinogram(y)
    n = geom.n_det
    h = np.zeros(n); h[0] = 0.25
    k = np.arange(1, n, 2); h[k] = -1.0 / (np.pi * k) ** 2
    H = h[np.abs(np.arange(n)[:, None] - np.arange(n)[None, :])]
    assert rel_l2(2 * np.pi / (2 * 90) * (y @ H.T), q) < 1e-12
    assert 0 < O.ramp_fourier_filter(128)[0] < 5e-3 and abs(O.ramp_fourier_filter(128)[64] - 1.0) < 5e-3   # ~2|xi|, small positive DC
    xx, yy = np.meshgrid(np.arange(64) - 31.5, np.arange(64) - 31.5, indexing='ij')
    x = ((xx / 20) ** 2 + (yy / 12) ** 2 < 1).astype(np.float32)[None]
    x = np.asarray(torch.nn.functional.avg_pool2d(torch.from_numpy(x)[None], 5, 1, 2)[0])
    rec = O.fbp(geom, O.fp(geom, x))
    assert rel_l2(rec, x) < 0.06
    assert abs(rec[0, 32, 32] - 1.0) < 0.02


def test_adaptation_loss_object_and_fused_objective_gate():
    """AdaptationLoss (the loss closure of get_standard_adapted_sampler as an object) evaluates the reference's
    expression; the fused objective only applies to the CUDA operator -- on CPU `_adapt` takes the tensor path."""
    from diffusion_models_dev_project_b200.samplers.adaptation import (AdaptationLoss, adapt_objective,
                                                                       adapt_objective_applies)
    from diffusion_models_dev_project_b200.samplers.utils import _AdaptGraph
    rt = _MatrixTrafo()
    g = torch.Generator().manual_seed(8)
    x = torch.rand(2, 1, 6, 5, generator=g)
    y = torch.rand(2, 1, 4, 7, generator=g)
    loss = AdaptationLoss(y, rt, 1e-2)
    ref = torch.mean((rt(x) - y).pow(2)) + 1e-2 * pkg.tv_loss(x)
    assert torch.equal(loss(x=x), ref) and torch.equal(loss(x), ref)
    sde = pkg.DDPM()
    assert not adapt_objective_applies(x, None, loss, sde, 'cg')                    # generic operator, CPU tensors
    assert adapt_objective(x.clone().requires_grad_(True), x, torch.ones(2), None, loss, sde, 0.1, 1, 'cg') is None
    assert not adapt_objective_applies(x, None, lambda x: x.sum(), sde, 'cg')
    # the graph cache key follows the observation (address and version), the operator and every scalar
    k1 = _AdaptGraph.make_key(loss, x, x, 1e-3, 0.1, 1, 'cg')
    assert k1 == _AdaptGraph.make_key(loss, x, x, 1e-3, 0.1, 1, 'cg')
    y.add_(1.0)
    assert k1 != _AdaptGraph.make_key(loss, x, x, 1e-3, 0.1, 1, 'cg')
    assert _AdaptGraph.make_key(loss, x, x, 1e-3, 0.1, 2, 'cg') != _AdaptGraph.make_key(loss, x, x, 1e-3, 0.1, 1, 'cg')


def test_bench_build_id_and_reference_arm_helpers():
    """bench.py records which library it measured (sha256 of the .so and of its sources) and how many host threads the
    CPU arm used."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    bid = bench.build_id()
    assert set(bid) == {'lib_sha16', 'src_sha16', 'stale'} and len(bid['lib_sha16']) == 16 and bid['stale'] is False
    assert bench.host_cores() >= 1
    pairs = bench.time_pairs()
    assert len(pairs) == 100 and pairs[0] == (990, 980) and pairs[-1] == (0, -1)


def test_bench_dump_outputs_float32_within_the_size_cap(tmp_path, monkeypatch):
    """--dump-outputs: one float32 .npy per returned array; above the cap the same seeded subset of samples is kept in
    every array, and the subset does not change from run to run."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = torch.arange(6 * 2 * 3, dtype=torch.float64).reshape(6, 1, 2, 3)
    bench.dump_outputs(str(tmp_path / 'full'), {'x_next': a, 'xhat0': -a})
    x, h = np.load(tmp_path / 'full' / 'x_next.npy'), np.load(tmp_path / 'full' / 'xhat0.npy')
    assert x.dtype == np.float32 and np.array_equal(x, a.numpy()) and np.array_equal(h, -a.numpy())
    monkeypatch.setattr(bench, 'DUMP_BYTES', 3 * 2 * 4 * 6)            # room for 3 of the 6 samples of both arrays
    for d in ('s1', 's2'):
        bench.dump_outputs(str(tmp_path / d), {'x_next': a, 'xhat0': -a}, rank=1, world=1)
    xs, hs = np.load(tmp_path / 's1' / 'x_next.npy'), np.load(tmp_path / 's1' / 'xhat0.npy')
    assert xs.shape == (3, 1, 2, 3) and np.array_equal(hs, -xs)
    assert np.array_equal(xs, np.load(tmp_path / 's2' / 'x_next.npy'))
    assert all(any(np.array_equal(r, s) for s in a.numpy()) for r in xs)
    bench.dump_outputs(str(tmp_path / 'r'), {'x_next': a}, rank=1, world=2)
    assert sorted(os.listdir(tmp_path / 'r')) == ['x_next_rank1.npy']
    monkeypatch.setattr(bench, 'DUMP_BYTES', 4 * 6 - 1)                 # not even one sample fits: refused
    with pytest.raises(AssertionError, match='dump limit'):
        bench.dump_outputs(str(tmp_path / 'e'), {'x_next': a})


def test_bench_reference_arm_honours_steps_and_dumps(tmp_path, monkeypatch, capsys):
    """--steps sets the number of timed steps of the CPU reference arm too (it is not clamped), --steps < 1 is
    refused, and --dump-outputs writes the arm's last (x_next, xhat0)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench_mod', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for bad in (['--steps', '0'], ['--warmup', '-1']):
        monkeypatch.setattr('sys.argv', ['bench.py'] + bad)
        with pytest.raises(SystemExit):
            bench.parse()
    calls = []
    arm = bench.cpu_reference_arm
    monkeypatch.setattr(bench, 'cpu_reference_arm', lambda a, s, w: calls.append((s, w)) or arm(a, s, w))
    monkeypatch.setattr('sys.argv', ['bench.py', '--impl', 'reference', '--unet', 'small', '--steps', '1', '--warmup',
                                     '2', '--dump-outputs', str(tmp_path)])
    capsys.readouterr()
    grad, threads = torch.is_grad_enabled(), torch.get_num_threads()
    try:
        bench.run_reference(bench.parse())
    finally:                                    # the arm switches autograd off and sets the thread count process-wide
        torch.set_grad_enabled(grad)
        torch.set_num_threads(threads)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert calls == [(1, 2)] and line['steps'] == 1 and line['warmup'] == 2
    for n in ('x_next', 'xhat0'):
        v = np.load(tmp_path / (n + '.npy'))
        assert v.shape == (1, 1, 256, 256) and v.dtype == np.float32 and np.isfinite(v).all()
