"""Limited-angle and non-uniform view sets on the GPU: weighted geometries (scd_geom_create_weighted) against the
weighted oracle, on every path the projector pair takes (batch 1: direct, 2: packed copy, 3 / 8 / 17: interleaved
groups of 4, 8 and 16), including wedges whose views all fall into one projector class and sets of 1-8 views.

  * public A, A* and normal_apply against the oracle;
  * all-ones weights: bit-identical to the unweighted geometry, same launches;
  * cg_solve / dds_step against the float64 reference of the weighted oracle matrices (per-sample time steps);
  * autograd pairing with per-view range cells, in float64 against the oracle matrices;
  * the fused adaptation objective against the tensor path differentiated by autograd;
  * fbp against the weighted oracle FBP."""
import dataclasses
from math import pi, sqrt

import numpy as np
import pytest
import torch

import angle_set_oracle as W
from conftest import rel_l2
from fp64_reference import TIME_PAIRS, time_steps
from oracle import oracle as O

pytestmark = pytest.mark.gpu

XHAT0_GATE = 1e-6
X_NEXT_GATE = 2e-5


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


def _G():
    from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D
    return ParallelBeamGeometry2D


def _golden(n):
    return np.mod(np.arange(n) * pi * (3.0 - sqrt(5.0)), pi)


def _sparse(n):
    """``n`` views spread over [0, pi) with a fixed jitter (non-uniform cells from 3 views on)."""
    jit = np.array([0.0, 0.31, -0.22, 0.17, -0.35, 0.08, 0.27, -0.13])[:n]
    return (np.arange(n) + 0.5 + jit) * (pi / n)


def _geometry(name, shape=(256, 256)):
    G = _G()
    if name == 'wedge90':
        return G.from_angle_range(shape, 60, 0.0, pi / 2)
    if name == 'wedge120':
        return G.from_angle_range(shape, 60, 0.0, 2 * pi / 3)
    if name == 'wedge_cls0':                      # |sin| > |cos| for every view: class 1 is empty
        return G.from_angle_range(shape, 60, pi / 3, 2 * pi / 3)
    if name == 'wedge_cls1':                      # every view class 1: class 0 is empty
        return G.from_angle_range(shape, 60, -pi / 6, pi / 6)
    if name.startswith('sparse'):
        return G.from_angles(shape, _sparse(int(name[6:])))
    if name == 'golden37':
        return G.from_angles(shape, _golden(37))
    if name == 'random60of180':
        keep = np.sort(np.random.default_rng(2024).choice(180, 60, replace=False))
        return G.from_angles(shape, (keep + 0.5) * (pi / 180))
    if name == 'wedge600_501':
        return G.from_angle_range((501, 501), 600, pi / 6, 2 * pi / 3)
    raise KeyError(name)


SETS = ['wedge90', 'wedge120', 'wedge_cls0', 'wedge_cls1', 'sparse1', 'sparse2', 'sparse3', 'sparse4', 'sparse8',
        'golden37', 'random60of180']
BATCHES = (1, 2, 3, 8, 17)


def _oracle(geom, adj_scale=None, weighted=True):
    return W.geometry(geom, adj_scale=adj_scale, weighted=weighted)


def _rt(geom):
    return _pkg().B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom)


def _phantoms(shape, n):
    from bench_support.phantoms import disk_ellipses
    return np.ascontiguousarray(disk_ellipses(n, shape[0], seed=11)[:, :, :shape[0], :shape[1]])


# ------------------------------------------------------------------------------------------ operators ---
def _check_operators(geom, batches):
    rt, og = _rt(geom), _oracle(geom)
    assert rt.adj_scale == geom.dphi
    gen = torch.Generator(device='cuda').manual_seed(1)
    for B in batches:
        x = torch.rand(B, 1, *geom.im_shape, device='cuda', generator=gen)
        y = rt(x)
        assert rel_l2(y.cpu().numpy(), O.fp(og, x.cpu().numpy())) < 1e-4, ('A', B)
        s = torch.randn(B, 1, *geom.obs_shape, device='cuda', generator=gen)
        z = rt.trafo_adjoint(s)
        assert rel_l2(z.cpu().numpy(), W.bp(og, s.cpu().numpy())) < 1e-4, ('A*', B)
        # the projector's interleaved output carries the weights: A*A composed without re-layout
        n = rt.normal_apply(x, 0.3)
        assert rel_l2(n.cpu().numpy(), (x + 0.3 * rt.trafo_adjoint(rt(x))).cpu().numpy()) < 1e-6, ('normal', B)


@pytest.mark.parametrize('name', SETS)
def test_operators_match_the_weighted_oracle(name):
    geom = _geometry(name)
    if name in ('wedge_cls0', 'wedge_cls1'):
        cls0 = np.abs(np.sin(geom.angles)) > np.abs(np.cos(geom.angles))
        assert cls0.all() if name == 'wedge_cls0' else not cls0.any()
    _check_operators(geom, BATCHES)


def test_operators_501_wedge_of_600_views():
    _check_operators(_geometry('wedge600_501'), (1, 3))


# ------------------------------------------------------------------------------------ unit weights ---
@pytest.mark.parametrize('batch', [1, 2, 8])
def test_unit_weights_are_the_unweighted_geometry(batch):
    pkg = _pkg()
    from diffusion_models_dev_project_b200 import fused
    base_geom = _G().from_im_shape((256, 256), 60)
    ones_geom = dataclasses.replace(base_geom, angle_weights=np.ones(60))
    a, b = _rt(base_geom), _rt(ones_geom)
    gen = torch.Generator(device='cuda').manual_seed(4)
    x, s, eps = (torch.randn(batch, 1, 256, 256, device='cuda', generator=gen) for _ in range(3))
    y = a(torch.rand(batch, 1, 256, 256, device='cuda', generator=gen))
    assert torch.equal(a.trafo_adjoint(y), b.trafo_adjoint(y))
    assert torch.equal(a.normal_apply(x, 0.2), b.normal_apply(x, 0.2))
    atb = a.trafo_adjoint(y)
    assert torch.equal(a.cg_solve(x, x + 0.01 * atb, 0.01, 5), b.cg_solve(x, x + 0.01 * atb, 0.01, 5))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    ra = a.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
    fused.launch_count(reset=True)
    rb = b.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
    n_launch = fused.launch_count()
    assert torch.equal(ra[0], rb[0]) and torch.equal(ra[1], rb[1])
    assert torch.equal(a.fbp(y), b.fbp(y))
    if batch == 8:
        assert n_launch == 19
    fused.launch_count(reset=True)
    a.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
    assert fused.launch_count() == n_launch


# ------------------------------------------------------------------------------- CG / DDS vs float64 ---
DC_CASES = [('wedge90', 8), ('wedge90', 2), ('golden37', 3), ('random60of180', 17), ('wedge_cls1', 1),
            ('sparse8', 8), ('wedge_cls0', 3)]


@pytest.mark.parametrize('name,batch', DC_CASES, ids=['%s-b%d' % c for c in DC_CASES])
def test_cg_and_dds_step_match_fp64_on_weighted_geometries(name, batch):
    """Gates of test_gpu_dds_step.py: xhat0 1e-6 and x_next 2e-5 per sample at gamma = 0.01, each sample with its
    own (t, t_prev).  The CG's internal sinogram must carry the view weights: without them the solve is the
    unweighted normal equation, percent-level away from the reference on these geometries."""
    pkg = _pkg()
    geom = _geometry(name)
    rt, og = _rt(geom), _oracle(geom)
    gen = torch.Generator(device='cuda').manual_seed(7)
    x, s, eps = (torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen) for _ in range(3))
    ph = torch.from_numpy(_phantoms(geom.im_shape, 4)[[b % 4 for b in range(batch)]]).cuda()
    atb = rt.trafo_adjoint(rt(ph))
    gamma, eta, n_iter = 0.01, 0.15, 5
    # CG alone
    x0, rhs = x, x + gamma * atb
    out = rt.cg_solve(x0, rhs, gamma, n_iter)
    ref = W.cg64(og, x0.cpu().numpy(), rhs.cpu().numpy(), gamma, n_iter)
    e = np.array([rel_l2(out[b].cpu().numpy(), ref[b]) for b in range(batch)])
    print('\ncg %s b%d: worst per-sample rel L2 vs fp64 %.2e' % (name, batch, e.max()))
    assert (e <= X_NEXT_GATE).all(), e
    # fused step
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch, TIME_PAIRS)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    x_next, xhat0 = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter)
    ref_next, ref_xh0 = W.dds_step64(og, x.cpu().numpy(), s.cpu().numpy(), atb.cpu().numpy(), eps.cpu().numpy(),
                                   t_np, tp_np, abar.cpu().numpy(), gamma, eta, n_iter)
    e_xh = np.array([rel_l2(xhat0[b].cpu().numpy(), ref_xh0[b]) for b in range(batch)])
    e_nx = np.array([rel_l2(x_next[b].cpu().numpy(), ref_next[b]) for b in range(batch)])
    print('dds_step %s b%d: worst per-sample rel L2 vs fp64: xhat0 %.2e, x_next %.2e' % (name, batch, e_xh.max(),
                                                                                          e_nx.max()))
    assert (e_xh <= XHAT0_GATE).all(), e_xh
    assert (e_nx <= X_NEXT_GATE).all(), e_nx


# --------------------------------------------------------------------------------------------- autograd ---
@pytest.mark.parametrize('name', ['wedge90', 'golden37'])
def test_autograd_pairing_with_per_view_cells(name):
    """d<g, A x>/dx = (dx^2/ds) BP_plain(g) (the unweighted transpose) and d<h, A* y>/dy = c_i (A h)_i with
    c_i = dphi w_i ds/dx^2, against the oracle matrices in float64."""
    geom = _geometry(name, (96, 96))
    rt = _rt(geom)
    J = O.joseph_matrix(_oracle(geom))
    Bplain = O.bp_matrix(_oracle(geom, adj_scale=1.0, weighted=False))
    gen = torch.Generator(device='cuda').manual_seed(9)
    B = 2
    x = torch.rand(B, 1, *geom.im_shape, device='cuda', generator=gen, requires_grad=True)
    g = torch.randn(B, 1, *geom.obs_shape, device='cuda', generator=gen)
    (rt(x) * g).sum().backward()
    g64 = g.cpu().numpy().reshape(B, -1).T.astype(np.float64)
    ref = (geom.dx ** 2 / geom.ds) * (Bplain @ g64)
    assert rel_l2(x.grad.cpu().numpy().reshape(B, -1).T, ref) < 1e-4
    y = torch.randn(B, 1, *geom.obs_shape, device='cuda', generator=gen, requires_grad=True)
    h = torch.rand(B, 1, *geom.im_shape, device='cuda', generator=gen)
    (rt.trafo_adjoint(y) * h).sum().backward()
    ah = (J @ h.cpu().numpy().reshape(B, -1).T.astype(np.float64)).T.reshape(B, 1, *geom.obs_shape)
    ref = ah * geom.range_weights[:, None]
    assert rel_l2(y.grad.cpu().numpy(), ref) < 1e-4


@pytest.mark.parametrize('dc_type', ['cg', 'gd'])
@pytest.mark.parametrize('n_iter', [1, 2])
@pytest.mark.parametrize('batch', [1, 3])
def test_fused_adaptation_objective_on_a_weighted_geometry(dc_type, n_iter, batch):
    """scd_adapt_fwd / scd_adapt_bwd on a golden-angle set against apTweedy -> cg | gradient step -> the loss
    written as a tensor expression, differentiated by autograd through trafo / trafo_adjoint."""
    pkg = _pkg()
    from diffusion_models_dev_project_b200.samplers.adaptation import AdaptationLoss, adapt_objective
    geom = _G().from_angles((64, 64), _golden(23))
    rt = _rt(geom)
    sde = pkg.DDPM()
    gen = torch.Generator(device='cuda').manual_seed(17)
    gt = torch.nn.functional.avg_pool2d(torch.rand(batch, 1, 64, 64, device='cuda', generator=gen), 5, 1, 2)
    y = rt(gt) + 0.01 * torch.randn(batch, 1, *rt.obs_shape, device='cuda', generator=gen)
    rhs = rt.trafo_adjoint(y)
    t = torch.ones(batch, device='cuda') * 300.
    ab = sde.alpha_bar_table('cuda')[301]
    x = ab.sqrt() * gt + (1 - ab).sqrt() * torch.randn(batch, 1, 64, 64, device='cuda', generator=gen)
    s0 = torch.randn(batch, 1, 64, 64, device='cuda', generator=gen)
    gamma, lam = 0.05, 1e-3
    loss_fn = AdaptationLoss(y, rt, lam)

    sa = s0.clone().requires_grad_(True)
    la = adapt_objective(sa, x, t, rhs, loss_fn, sde, gamma, n_iter, dc_type)
    assert la is not None
    (3.0 * la).backward()

    sb = s0.clone().requires_grad_(True)
    xhat0 = pkg.apTweedy(s=sb, x=x, sde=sde, time_step=t)
    if dc_type == 'cg':
        xhat = pkg.cg(op=rt.normal_op(gamma), x=xhat0, rhs=xhat0 + gamma * rhs, n_iter=n_iter)
    else:
        xhat = xhat0 - gamma * rt.trafo_adjoint(rt(xhat0)) + gamma * rhs
    lb = torch.mean((rt(xhat) - y).pow(2)) + lam * pkg.tv_loss(xhat)
    (3.0 * lb).backward()
    assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-5, (float(la), float(lb))
    assert rel_l2(sa.grad.cpu().numpy(), sb.grad.cpu().numpy()) < 1e-4
    # the fused data-fit loss (adaptation_loss) has the same gradient
    xa = xhat.detach().clone().requires_grad_(True)
    pkg.adaptation_loss(xa, y, rt, lam).backward()
    xb = xhat.detach().clone().requires_grad_(True)
    (torch.mean((rt(xb) - y).pow(2)) + lam * pkg.tv_loss(xb)).backward()
    assert rel_l2(xa.grad.cpu().numpy(), xb.grad.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------- fbp ---
@pytest.mark.parametrize('name', ['wedge90', 'golden37', 'random60of180'])
def test_fbp_matches_the_weighted_oracle_fbp(name):
    geom = _geometry(name)
    rt, og = _rt(geom), _oracle(geom)
    x = torch.from_numpy(_phantoms(geom.im_shape, 2)).cuda()
    y = rt(x)
    out = rt.fbp(y).cpu().numpy()
    ref = W.fbp(og, y.cpu().numpy())
    assert rel_l2(out, ref) < 1e-4
