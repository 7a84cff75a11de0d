"""Measurement weights W on the B200 (penalised weighted least squares): op(v) = v + gamma A*(W A v) through
normal_apply, the fused CG, the fused DDS step and the fused SCD adaptation objective.

  * W = 1 gives the same bits as no weights on every batch path (1: the caller's tensors, 2: packed copies, 3 / 8 /
    16 / 17 / 40: interleaved groups), and a broadcast [n_angles, n_det] weight the bits of its expanded copy;
  * per-sample weights over three orders of magnitude, with zeroed views and bins, against the float64 oracle of
    tests/stat_weights_oracle.py (uniform, 96 x 70, 501^2, a wedge, a golden-angle set, the matched adjoint);
  * the fused adaptation objective against its tensor expression differentiated by autograd;
  * a CUDA-graph capture of a weighted DDS step replays identically, and no call writes its inputs;
  * weights per sample and channel ([B, C, ...] and broadcasts of it), a private copy of W, packed copies that follow
    the launch tuning, and factories that validate and pack W once for the whole sampling run.
"""
import numpy as np
import pytest
import torch

import angle_set_oracle as AO
import stat_weights_oracle as SW
import test_gpu_angle_sets as AS
from conftest import rel_l2
from fp64_reference import TIME_PAIRS, time_steps

pytestmark = pytest.mark.gpu

NORMAL_GATE = 1e-5
CG_GATE = 1e-5
X_NEXT_GATE = 2e-5
BATCHES = [1, 2, 3, 8, 16, 17, 40]


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


def _G():
    from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D
    return ParallelBeamGeometry2D


def _geometry(name):
    shapes = {'u256': ((256, 256), 60), 'u96x70': ((96, 70), 18), 'u501': ((501, 501), 60), 'u64': ((64, 64), 23)}
    if name in shapes:
        return _G().from_im_shape(*shapes[name])
    return AS._geometry(name)


def _rt(geom, adjoint='pixel'):
    return _pkg().B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom, adjoint=adjoint)


def _per_sample(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    return np.array([rel_l2(a[i], b[i]) for i in range(a.shape[0])])


def _stat_weights(batch, obs_shape, seed):
    """Per-sample weights 10^U(-1.5, 1.5), mean 1 per sample, with one zeroed view and a few zeroed bins each."""
    rng = np.random.default_rng(seed)
    w = 10.0 ** rng.uniform(-1.5, 1.5, size=(batch, 1, *obs_shape))
    for b in range(batch):
        w[b, 0, rng.integers(obs_shape[0])] = 0.0
        w[b, 0, :, rng.integers(obs_shape[1], size=5)] = 0.0
    w /= w.reshape(batch, -1).mean(1)[:, None, None, None]
    return torch.from_numpy(w).float().cuda()


def _inputs(geom, batch, seed=7):
    gen = torch.Generator(device='cuda').manual_seed(seed)
    return [torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen) for _ in range(3)]


# ------------------------------------------------------------------------------------------ bit-identity ---
@pytest.mark.parametrize('batch', BATCHES)
def test_unit_weights_give_the_unweighted_bits(batch):
    pkg = _pkg()
    geom = _geometry('u256')
    rt = _rt(geom)
    x, s, eps = _inputs(geom, batch)
    y = rt(torch.nn.functional.avg_pool2d(x.abs(), 5, 1, 2))
    atb = rt.trafo_adjoint(y)
    ones = torch.ones(*rt.obs_shape, device='cuda')
    gamma, eta, n_iter = 0.01, 0.15, 5
    assert torch.equal(rt.normal_apply(x, gamma, weights=ones), rt.normal_apply(x, gamma))
    assert torch.equal(rt.cg_solve(x, x + gamma * atb, gamma, n_iter, weights=ones),
                       rt.cg_solve(x, x + gamma * atb, gamma, n_iter))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch, TIME_PAIRS)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    a = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter, weights=ones)
    b = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # a broadcast weight map and its per-sample copy
    w2 = _stat_weights(1, rt.obs_shape, 5)[0, 0]
    wb = w2.expand(batch, 1, *rt.obs_shape).contiguous()
    assert torch.equal(rt.normal_apply(x, gamma, weights=w2), rt.normal_apply(x, gamma, weights=wb))
    assert torch.equal(rt.cg_solve(x, x, gamma, n_iter, weights=w2), rt.cg_solve(x, x, gamma, n_iter, weights=wb))
    a = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter, weights=w2)
    b = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter, weights=wb)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # the fused adaptation objective (forward loss and the whole reverse sweep)
    from diffusion_models_dev_project_b200.samplers.adaptation import AdaptationLoss, adapt_objective
    sde = pkg.DDPM()
    tt = torch.full((batch,), 300., device='cuda')
    for dc in ('cg', 'gd', 'none'):
        out = []
        for w in (None, ones):
            sg = s.clone().requires_grad_(True)
            loss = adapt_objective(sg, x, tt, atb, AdaptationLoss(y, rt, 1e-3, weights=w), sde, gamma, 2, dc)
            loss.backward()
            out.append((loss.detach(), sg.grad))
        assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), dc


# ------------------------------------------------------------------------------------ accuracy vs float64 ---
ACC_CASES = [('u256', b, 'pixel') for b in BATCHES] + [
    ('u96x70', 8, 'pixel'), ('u501', 1, 'pixel'), ('wedge90', 8, 'pixel'), ('golden37', 3, 'pixel'),
    ('u256', 8, 'matched'), ('golden37', 2, 'matched')]


@pytest.mark.parametrize('name,batch,adjoint', ACC_CASES, ids=['%s-b%d-%s' % c for c in ACC_CASES])
def test_weighted_system_matches_fp64(name, batch, adjoint):
    pkg = _pkg()
    geom = _geometry(name)
    rt, og = _rt(geom, adjoint), AO.geometry(geom)
    J, Bm = SW.matrices(og, adjoint)
    x, s, eps = _inputs(geom, batch)
    w = _stat_weights(batch, rt.obs_shape, 11)
    w_np = w.cpu().numpy()
    gamma, eta, n_iter = 0.01, 0.15, 5
    e_n = _per_sample(rt.normal_apply(x, gamma, weights=w), SW.normal64(J, Bm, og, x.cpu().numpy(), gamma, w_np))
    y = rt(torch.nn.functional.avg_pool2d(x.abs(), 5, 1, 2))
    atb = rt.trafo_adjoint(w * y)
    rhs = x + gamma * atb
    e_cg = _per_sample(rt.cg_solve(x, rhs, gamma, n_iter, weights=w),
                       SW.cg64(J, Bm, og, x.cpu().numpy(), rhs.cpu().numpy(), gamma, n_iter, w_np))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch, TIME_PAIRS)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    x_next, xhat0 = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter, weights=w)
    ref_next, _ = SW.dds_step64(J, Bm, og, x.cpu().numpy(), s.cpu().numpy(), atb.cpu().numpy(), eps.cpu().numpy(),
                                t_np, tp_np, abar.cpu().numpy(), gamma, eta, n_iter, w_np)
    e_nx = _per_sample(x_next, ref_next)
    print('\n%s b%d %s: normal %.2e  cg %.2e  dds x_next %.2e' % (name, batch, adjoint, e_n.max(), e_cg.max(), e_nx.max()))
    assert (e_n <= NORMAL_GATE).all(), e_n
    assert (e_cg <= CG_GATE).all(), e_cg
    assert (e_nx <= X_NEXT_GATE).all(), e_nx


# -------------------------------------------------------------------------------------------- adaptation ---
@pytest.mark.parametrize('dc_type', ['cg', 'gd', 'none'])
@pytest.mark.parametrize('batch', [1, 3])
def test_fused_adaptation_with_weights_matches_autograd(dc_type, batch):
    pkg = _pkg()
    from diffusion_models_dev_project_b200.samplers.adaptation import AdaptationLoss, adapt_objective
    for geom, adjoint in ((_geometry('u64'), 'pixel'), (_G().from_angles((64, 64), AS._golden(23)), 'matched')):
        rt = _rt(geom, adjoint)
        sde = pkg.DDPM()
        gen = torch.Generator(device='cuda').manual_seed(17)
        gt = torch.nn.functional.avg_pool2d(torch.rand(batch, 1, 64, 64, device='cuda', generator=gen), 5, 1, 2)
        y = rt(gt) + 0.01 * torch.randn(batch, 1, *rt.obs_shape, device='cuda', generator=gen)
        w = _stat_weights(batch, rt.obs_shape, 23)
        rhs = rt.trafo_adjoint(w * y)
        t = torch.ones(batch, device='cuda') * 300.
        ab = sde.alpha_bar_table('cuda')[301]
        x = ab.sqrt() * gt + (1 - ab).sqrt() * torch.randn(batch, 1, 64, 64, device='cuda', generator=gen)
        s0 = torch.randn(batch, 1, 64, 64, device='cuda', generator=gen)
        gamma, lam, n_iter = 0.05, 1e-3, 2
        sa = s0.clone().requires_grad_(True)
        la = adapt_objective(sa, x, t, rhs, AdaptationLoss(y, rt, lam, weights=w), sde, gamma, n_iter, dc_type)
        assert la is not None
        (3.0 * la).backward()
        # the tensor expression through trafo / trafo_adjoint, differentiated by autograd (a plain callable: cg
        # runs its tensor recurrences)
        sb = s0.clone().requires_grad_(True)
        xhat0 = pkg.apTweedy(s=sb, x=x, sde=sde, time_step=t)
        if dc_type == 'cg':
            xhat = pkg.cg(op=lambda v: v + gamma * rt.trafo_adjoint(w * rt(v)), x=xhat0, rhs=xhat0 + gamma * rhs,
                          n_iter=n_iter)
        elif dc_type == 'gd':
            xhat = xhat0 - gamma * rt.trafo_adjoint(w * rt(xhat0)) + gamma * rhs
        else:
            xhat = xhat0
        lb = torch.mean(w * (rt(xhat) - y).pow(2)) + lam * pkg.tv_loss(xhat)
        (3.0 * lb).backward()
        assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-4, (float(la), float(lb))
        assert rel_l2(sa.grad.cpu().numpy(), sb.grad.cpu().numpy()) < 1e-4


def test_weighted_adaptation_loss_matches_its_expression():
    """adaptation_loss with weights (scd_residual_sq_w forward, one backprojection backward) against autograd."""
    pkg = _pkg()
    rt = _rt(_geometry('u64'))
    gen = torch.Generator(device='cuda').manual_seed(3)
    xa = torch.rand(3, 1, 64, 64, device='cuda', generator=gen).requires_grad_(True)
    xb = xa.detach().clone().requires_grad_(True)
    y = rt(torch.rand(3, 1, 64, 64, device='cuda', generator=gen))
    w = _stat_weights(3, rt.obs_shape, 2)
    la = pkg.adaptation_loss(xa, y, rt, 1e-3, weights=w)
    la.backward()
    lb = torch.mean(w * (rt(xb) - y).pow(2)) + 1e-3 * pkg.tv_loss(xb)
    lb.backward()
    assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-5
    assert rel_l2(xa.grad.cpu().numpy(), xb.grad.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------- capture, untouched inputs ---
@pytest.mark.parametrize('batch', [1, 2, 8])
def test_weighted_dds_step_captures_and_leaves_inputs_alone(batch):
    pkg = _pkg()
    geom = _geometry('u256')
    rt = _rt(geom)
    x, s, eps = _inputs(geom, batch)
    w = _stat_weights(batch, rt.obs_shape, 4)
    y = rt(torch.nn.functional.avg_pool2d(x.abs(), 5, 1, 2))
    atb = rt.trafo_adjoint(w * y)
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch, TIME_PAIRS)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    mw = pkg.MeasurementWeights(rt, w)
    before = [v.clone() for v in (x, s, atb, eps, t, tp, w, y)]
    eager = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5, weights=mw)     # packs W (outside the capture)
    rt.normal_apply(x, 0.01, weights=mw)
    rt.cg_solve(x, atb, 0.01, 5, weights=mw)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5, weights=mw)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(captured[0], eager[0]) and torch.equal(captured[1], eager[1])
    for a, b in zip(before, (x, s, atb, eps, t, tp, w, y)):
        assert torch.equal(a, b)


def test_rejections_on_the_device():
    pkg = _pkg()
    rt = _rt(_geometry('u64'))
    x = torch.zeros(3, 1, 64, 64, device='cuda')
    with pytest.raises(ValueError, match='do not broadcast'):
        rt.normal_apply(x, 0.1, weights=torch.ones(2, 1, *rt.obs_shape, device='cuda'))
    other = _rt(_geometry('u64'))
    with pytest.raises(ValueError, match='another ray transform'):
        rt.cg_solve(x, x, 0.1, 2, weights=pkg.MeasurementWeights(other, torch.ones(*rt.obs_shape, device='cuda')))


# ------------------------------------------------------------------------- shapes, copies, tuning, factories ---
def test_weights_per_sample_and_channel():
    """[B, C, ...] weights on [B, C, ...] observations are the flattened [B*C, 1, ...] case; [B, 1, ...] broadcasts
    over the channels like its expanded copy."""
    pkg = _pkg()
    geom = _geometry('u64')
    rt = _rt(geom)
    gen = torch.Generator(device='cuda').manual_seed(9)
    x, s, eps = (torch.randn(2, 3, 64, 64, device='cuda', generator=gen) for _ in range(3))
    w = _stat_weights(6, rt.obs_shape, 8).reshape(2, 3, *rt.obs_shape)
    flat = lambda a: a.reshape(6, 1, *a.shape[-2:])                 # noqa: E731
    atb = rt.trafo_adjoint(w * rt(x.abs()))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t, tp = torch.full((6,), 500., device='cuda'), torch.full((6,), 490., device='cuda')
    assert torch.equal(flat(rt.normal_apply(x, 0.05, weights=w)), rt.normal_apply(flat(x), 0.05, weights=flat(w)))
    assert torch.equal(flat(rt.cg_solve(x, atb, 0.05, 4, weights=w)),
                       rt.cg_solve(flat(x), flat(atb), 0.05, 4, weights=flat(w)))
    a = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.05, 0.15, 4, weights=w)
    b = rt.dds_step(flat(x), flat(s), flat(atb), flat(eps), t, tp, abar, 0.05, 0.15, 4, weights=flat(w))
    assert torch.equal(flat(a[0]), b[0]) and torch.equal(flat(a[1]), b[1])
    w1 = w[:, :1].contiguous()
    assert torch.equal(rt.normal_apply(x, 0.05, weights=w1),
                       rt.normal_apply(x, 0.05, weights=w1.expand(2, 3, *rt.obs_shape).contiguous()))
    with pytest.raises(ValueError, match='broadcast'):
        rt.normal_apply(x, 0.05, weights=w[:, :2].contiguous())


def test_weights_are_a_private_copy():
    """Changing the caller's tensor after the weights were made changes neither the fused nor the tensor path."""
    pkg = _pkg()
    rt = _rt(_geometry('u64'))
    x = torch.randn(3, 1, 64, 64, device='cuda', generator=torch.Generator(device='cuda').manual_seed(1))
    w = _stat_weights(3, rt.obs_shape, 6)
    mw = pkg.MeasurementWeights(rt, w)
    before = rt.normal_apply(x, 0.05, weights=mw)
    w.mul_(2.0)
    assert torch.equal(rt.normal_apply(x, 0.05, weights=mw), before)
    xg = x.clone().requires_grad_(True)
    tensor_path = pkg.NormalOp(rt, 0.05, mw)(xg)                     # trafo / trafo_adjoint expression
    assert rel_l2(tensor_path.detach().cpu().numpy(), before.cpu().numpy()) < 1e-6


def test_packed_weights_follow_the_launch_tuning():
    pkg = _pkg()
    rt = _rt(_geometry('u256'))
    x = torch.randn(8, 1, 256, 256, device='cuda', generator=torch.Generator(device='cuda').manual_seed(2))
    w = _stat_weights(8, rt.obs_shape, 7)
    mw = pkg.MeasurementWeights(rt, w)
    ref = rt.normal_apply(x, 0.01, weights=mw)
    try:
        rt.set_tuning('cuda', fp_samples=4)                          # groups of 4 instead of 8: another layout
        tuned = rt.normal_apply(x, 0.01, weights=mw)
        fresh = rt.normal_apply(x, 0.01, weights=pkg.MeasurementWeights(rt, w))
        assert torch.equal(tuned, fresh)
        assert rel_l2(tuned.cpu().numpy(), ref.cpu().numpy()) < 1e-6
        assert len([k for k in mw._cache if k[0] == 'il']) == 1     # the copy of the earlier tuning is dropped
    finally:
        rt.set_tuning('cuda', fp_samples=0)


def test_factories_validate_and_pack_once(monkeypatch):
    """The standard samplers hand their predictors one MeasurementWeights: the sampling steps neither validate nor
    pack the weights again.  A MeasurementWeights given to a factory is used as it is."""
    pkg = _pkg()
    from types import SimpleNamespace as NS
    from diffusion_models_dev_project_b200 import _lib
    geom = _geometry('u64')
    rt = _rt(geom)
    batch = 2
    gen = torch.Generator(device='cuda').manual_seed(5)
    y = rt(torch.rand(batch, 1, 64, 64, device='cuda', generator=gen))
    w = _stat_weights(batch, rt.obs_shape, 12)
    args = NS(method='dds', num_steps=4, pct_chain_elapsed=0, eta=0.15, gamma=0.02, cg_iter=3, adaptation='full',
              num_optim_step=1, adapt_freq=1, lr=1e-3, tv_penalty=1e-4, add_cg=True, dc_type='cg',
              early_stopping_pct=1.0)
    config = NS(device='cuda', sampling=NS(batch_size=batch, eps=1e-3, travel_length=1, travel_repeat=1),
                model=NS(in_channels=1))
    score = lambda x, t: 0.1 * x                                      # noqa: E731
    sde = pkg.DDPM()
    sampler = pkg.get_standard_sampler(args, config, score, sde, rt, observation=y, weights=w)
    mw = sampler.predictor.keywords['cg_kwargs']['weights']
    assert isinstance(mw, pkg.MeasurementWeights)
    assert torch.equal(sampler.predictor.keywords['rhs'], rt.trafo_adjoint(w * y))
    made, packs = [0], [0]
    init = pkg.MeasurementWeights.__init__
    lib = _lib.load()
    pack = lib.scd_sino_weights_pack

    def counting_init(self, *a, **k):
        made[0] += 1
        init(self, *a, **k)

    def counting_pack(*a):
        packs[0] += 1
        return pack(*a)
    monkeypatch.setattr(pkg.MeasurementWeights, '__init__', counting_init)
    monkeypatch.setattr(lib, 'scd_sino_weights_pack', counting_pack)
    x = torch.randn(batch, 1, 64, 64, device='cuda', generator=gen)
    for k in range(3):
        t = torch.full((batch,), 500. - 10 * k, device='cuda')
        x, _ = sampler.predictor(score=score, sde=sde, x=x, time_step=(t, t - 10), step_size=1.0,
                                 **sampler.sample_kwargs['predictor'])
    assert torch.isfinite(x).all()
    assert made[0] == 0 and packs[0] == 1, (made, packs)
    monkeypatch.undo()
    # a MeasurementWeights given to the factories
    mw2 = pkg.MeasurementWeights(rt, w)
    sampler = pkg.get_standard_sampler(args, config, score, sde, rt, observation=y, weights=mw2)
    assert sampler.predictor.keywords['cg_kwargs']['weights'] is mw2
    assert torch.equal(sampler.predictor.keywords['rhs'], rt.trafo_adjoint(w * y))
    sampler = pkg.get_standard_adapted_sampler(args, config, torch.nn.Conv2d(1, 1, 1).cuda(), sde, rt, observation=y,
                                               weights=mw2)
    kw = sampler.predictor.keywords
    assert kw['cg_kwargs']['weights'] is mw2 and kw['adapt_fn'].keywords['loss_fn'].weights is mw2
    assert torch.equal(kw['rhs'], rt.trafo_adjoint(w * y))
