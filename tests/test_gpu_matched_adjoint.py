"""The matched adjoint on the GPU (``B200RayTrafo(adjoint='matched')``, scd_geom_create_ex with
SCD_GEOM_MATCHED_ADJOINT): every backprojection the library launches against the float64 transpose of the Joseph
matrix, ``c_w J^T diag(w)`` (tests/matched_adjoint_oracle.py).

  * A* per sample within 1e-5 on every batch path (1: direct, 2: packed, 3 / 8 / 16 / 17 / 40: groups of 4, 8, 16),
    the tile heights 8 / 16 / 32 with the pair march on and off (bit-identical), four image shapes, weighted view
    sets, angle ranges, and the host-buffer entry point;
  * the dot test and the symmetry of ``I + gamma A*A`` (the pixel-driven pair is >= 100x further off);
  * cg_solve / dds_step against the float64 recurrences on (J, c_w J^T) with the gates of test_gpu_dds_step.py;
  * autograd: the gradient through ``trafo`` is J^T g, and the reference's DPS / EM-DPS / Langevin goldens (built on
    torch.sparse, i.e. the exact transpose) are reproduced;
  * the fused adaptation objective against the autograd tensor path;
  * the peer-staged banded backprojection for 1 to 8 emulated ranks;
  * fbp against its matched oracle;
  * rejection of dx/ds >= 1.5 and of unknown flag bits."""
import ctypes as C

import numpy as np
import pytest
import torch

import angle_set_oracle as W
import banded_emulation as E
import matched_adjoint_oracle as M
import test_gpu_angle_sets as AS
import test_gpu_banded as TB
from conftest import rel_l2
from fp64_reference import TIME_PAIRS, time_steps

pytestmark = pytest.mark.gpu

BP_GATE = 1e-5
XHAT0_GATE = 1e-6
X_NEXT_GATE = 2e-5


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


def _G():
    from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D
    return ParallelBeamGeometry2D


def _geometry(name):
    shapes = {'u256': ((256, 256), 60), 'u96x70': ((96, 70), 18), 'u70x50': ((70, 50), 30),
              'u501': ((501, 501), 1200), 'u24': ((24, 24), 8), 'u64': ((64, 64), 23)}
    if name in shapes:
        return _G().from_im_shape(*shapes[name])
    return AS._geometry(name)


def _rt(geom, adjoint='matched'):
    return _pkg().B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom, adjoint=adjoint)


def _per_sample(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else a
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else b
    return np.array([rel_l2(a[i], b[i]) for i in range(a.shape[0])])


def _noise(shape, seed):
    return torch.randn(*shape, device='cuda', generator=torch.Generator(device='cuda').manual_seed(seed))


# ------------------------------------------------------------------------------------------------- A* ---
@pytest.mark.parametrize('batch', [1, 2, 3, 8, 16, 17, 40])
def test_matched_bp_every_batch_path(batch):
    geom = _geometry('u256')
    rt, og = _rt(geom), W.geometry(geom)
    y = _noise((batch, 1, *geom.obs_shape), batch)
    e = _per_sample(rt.trafo_adjoint(y), M.bp64(og, y.cpu().numpy()))
    print('\nA* matched 256^2/60 B=%d: worst per-sample rel L2 vs fp64 %.2e' % (batch, e.max()))
    assert (e <= BP_GATE).all(), e
    # the default operator is the pixel-driven one, percent-level away from the transpose on white noise
    assert (_per_sample(_rt(geom, 'pixel').trafo_adjoint(y), M.bp64(og, y.cpu().numpy())) > 1e-2).all()


@pytest.mark.parametrize('batch', [1, 8, 16])
@pytest.mark.parametrize('tile', [8, 16, 32])
def test_tile_heights_and_the_pair_march(tile, batch):
    """The pair march (3 loads per pixel pair on 2-tap views) is bit-identical to the plain matched march."""
    geom = _geometry('u256')
    rt, og = _rt(geom), W.geometry(geom)
    y = _noise((batch, 1, *geom.obs_shape), 10 + batch)
    ref = M.bp64(og, y.cpu().numpy())
    rt.set_tuning('cuda', bp_tile=tile, bp_rows=1)
    shared = rt.trafo_adjoint(y)
    rt.set_tuning('cuda', bp_share=1)
    plain = rt.trafo_adjoint(y)
    assert torch.equal(shared, plain)
    e = _per_sample(shared, ref)
    print('\nA* matched tile %d B=%d: %.2e' % (tile, batch, e.max()))
    assert (e <= BP_GATE).all(), e


@pytest.mark.parametrize('name,batches', [('u96x70', (1, 3, 8)), ('u70x50', (1, 2, 17)), ('wedge90', (1, 3, 8)),
                                          ('golden37', (1, 2, 8)), ('sparse3', (1, 3, 17))])
def test_matched_bp_shapes_and_view_sets(name, batches):
    geom = _geometry(name)
    rt, og = _rt(geom), W.geometry(geom)
    for B in batches:
        y = _noise((B, 1, *geom.obs_shape), B)
        e = _per_sample(rt.trafo_adjoint(y), M.bp64(og, y.cpu().numpy()))
        print('\nA* matched %s B=%d: %.2e' % (name, B, e.max()))
        assert (e <= BP_GATE).all(), (B, e)


def test_matched_bp_501_of_1200_views():
    """Two slices of a 501^2 x 1200-view stack, against the float64 hat restatement (tests/test_matched_adjoint_cpu.py
    shows it is c_w J^T to 1e-12) on every 7th image row."""
    geom = _geometry('u501')
    rt, og = _rt(geom), W.geometry(geom)
    y = _noise((2, 1, *geom.obs_shape), 501)
    rows = np.arange(0, 501, 7)
    out = rt.trafo_adjoint(y)[:, :, rows].cpu().numpy()
    e = _per_sample(out, M.bp_hat64(og, y.cpu().numpy(), rows=rows))
    print('\nA* matched 501^2/1200: %.2e' % e.max())
    assert (e <= BP_GATE).all(), e


@pytest.mark.parametrize('name', ['u256', 'golden37'])
def test_matched_bp_of_angle_ranges(name):
    geom = _geometry(name)
    rt, og = _rt(geom), W.geometry(geom)
    y = _noise((8, 1, *geom.obs_shape), 3)
    na = geom.n_angles
    for lo, hi in ((0, na // 3), (na // 3, na - 5), (na - 1, na), (7, 8)):
        ym = y.clone()
        ym[..., :lo, :] = 0
        ym[..., hi:, :] = 0
        e = _per_sample(rt._bp(y, rt.adj_scale, angle_range=(lo, hi)), M.bp64(og, ym.cpu().numpy()))
        assert (e <= BP_GATE).all(), (lo, hi, e)


def test_host_buffer_entry_point():
    geom = _geometry('u96x70')
    rt, og = _rt(geom), W.geometry(geom)
    y = np.random.default_rng(2).standard_normal((2, *geom.obs_shape)).astype(np.float32)
    z = np.zeros((2, *geom.im_shape), dtype=np.float32)
    h = rt._handle(torch.device('cuda'))
    from diffusion_models_dev_project_b200 import _lib
    _lib.check(h._lib.scd_bp_host(h.ptr, y.ctypes.data, z.ctypes.data, 2), 'scd_bp_host')
    assert (_per_sample(z, M.bp64(og, y)) <= BP_GATE).all()


# ------------------------------------------------------------------------------------ dot test, symmetry ---
def _phantoms(shape, n, seed=11):
    from bench_support.phantoms import disk_ellipses
    return torch.from_numpy(np.ascontiguousarray(disk_ellipses(n, shape[0], seed=seed)[:, :, :shape[0], :shape[1]])).cuda()


@pytest.mark.parametrize('name', ['u256', 'u96x70', 'golden37'])
def test_dot_test(name):
    """``|<Ax, y> - <x, A*y>/c_i|`` over ``||Ax|| ||y||`` (its Cauchy-Schwarz bound), on white-noise images and
    sinograms, with the per-view cells ``c_i = c_w w_i`` carried by A*.  The pixel-driven pair is >= 100x further off."""
    geom = _geometry(name)
    x = _noise((4, 1, *geom.im_shape), 40)
    y = _noise((4, 1, *geom.obs_shape), 41)
    yw = (y / torch.as_tensor(geom.view_weights, dtype=torch.float32, device='cuda')[:, None]).contiguous()
    gaps = {}
    for adjoint in ('matched', 'pixel'):
        rt = _rt(geom, adjoint)
        ax = rt(x).double()
        aty = rt.trafo_adjoint(yw).double() / geom.range_weight
        lhs = (ax * y.double()).sum(dim=(1, 2, 3))
        rhs = (x.double() * aty).sum(dim=(1, 2, 3))
        scale = ax.flatten(1).norm(dim=1) * y.double().flatten(1).norm(dim=1)
        gaps[adjoint] = ((lhs - rhs).abs() / scale).cpu().numpy()
    print('\ndot test %s: matched %.2e, pixel %.2e' % (name, gaps['matched'].max(), gaps['pixel'].min()))
    assert (gaps['matched'] <= 1e-5).all(), gaps
    assert gaps['pixel'].min() >= 100 * gaps['matched'].max(), gaps


@pytest.mark.parametrize('batch', [1, 8])
def test_normal_operator_is_symmetric(batch):
    geom = _geometry('u256')
    rt = _rt(geom)
    gen = torch.Generator(device='cuda').manual_seed(21)
    u = torch.rand(batch, 1, *geom.im_shape, device='cuda', generator=gen)
    v = torch.rand(batch, 1, *geom.im_shape, device='cuda', generator=gen)
    for gamma in (0.01, 1.0):
        a = (u.double() * rt.normal_apply(v, gamma).double()).sum(dim=(1, 2, 3))
        b = (rt.normal_apply(u, gamma).double() * v.double()).sum(dim=(1, 2, 3))
        gap = ((a - b).abs() / a.abs()).cpu().numpy()
        print('\nsymmetry B=%d gamma=%g: %.2e' % (batch, gamma, gap.max()))
        assert (gap <= 1e-6).all(), gap
        # the matched normal operator itself, against float64
        e = _per_sample(rt.normal_apply(v, gamma), M.normal64(W.geometry(geom), v.cpu().numpy(), gamma))
        assert (e <= BP_GATE).all(), e


# ------------------------------------------------------------------------------------ CG / DDS vs float64 ---
DC_CASES = [('u256', 1), ('u256', 2), ('u256', 3), ('u256', 8), ('u256', 17), ('u96x70', 8), ('golden37', 3)]


@pytest.mark.parametrize('name,batch', DC_CASES, ids=['%s-b%d' % c for c in DC_CASES])
def test_cg_and_dds_step_match_fp64(name, batch):
    """Batch 1: the caller's tensors; 2: packed copies; 3 / 8 / 17: interleaved groups of 4, 8 and 16."""
    pkg = _pkg()
    geom = _geometry(name)
    rt, og = _rt(geom), W.geometry(geom)
    gen = torch.Generator(device='cuda').manual_seed(7)
    x, s, eps = (torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen) for _ in range(3))
    ph = _phantoms(geom.im_shape, 4)[[b % 4 for b in range(batch)]]
    atb = rt.trafo_adjoint(rt(ph))
    gamma, eta, n_iter = 0.01, 0.15, 5
    out = rt.cg_solve(x, x + gamma * atb, gamma, n_iter)
    e = _per_sample(out, M.cg64(og, x.cpu().numpy(), (x + gamma * atb).cpu().numpy(), gamma, n_iter))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t_np, tp_np = time_steps(batch, TIME_PAIRS)
    t, tp = torch.from_numpy(t_np).cuda(), torch.from_numpy(tp_np).cuda()
    x_next, xhat0 = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter)
    ref_next, ref_xh0 = M.dds_step64(og, x.cpu().numpy(), s.cpu().numpy(), atb.cpu().numpy(), eps.cpu().numpy(),
                                     t_np, tp_np, abar.cpu().numpy(), gamma, eta, n_iter)
    e_xh, e_nx = _per_sample(xhat0, ref_xh0), _per_sample(x_next, ref_next)
    print('\n%s b%d: cg %.2e, dds_step xhat0 %.2e x_next %.2e' % (name, batch, e.max(), e_xh.max(), e_nx.max()))
    assert (e <= X_NEXT_GATE).all(), e
    assert (e_xh <= XHAT0_GATE).all(), e_xh
    assert (e_nx <= X_NEXT_GATE).all(), e_nx


# --------------------------------------------------------------------------------------------- autograd ---
@pytest.mark.parametrize('name', ['u64', 'u96x70', 'golden37'])
def test_gradient_through_trafo_is_the_transpose(name):
    geom = _geometry(name) if name != 'golden37' else _G().from_angles((64, 64), AS._golden(37))
    rt, og = _rt(geom), W.geometry(geom)
    B = 3
    gen = torch.Generator(device='cuda').manual_seed(9)
    x = torch.rand(B, 1, *geom.im_shape, device='cuda', generator=gen, requires_grad=True)
    g = torch.randn(B, 1, *geom.obs_shape, device='cuda', generator=gen)
    (rt(x) * g).sum().backward()
    J = M.joseph(og)
    ref = (J.T @ g.cpu().numpy().reshape(B, -1).T.astype(np.float64)).T.reshape(B, 1, *geom.im_shape)
    e = _per_sample(x.grad, ref)
    print('\ngrad of <g, A x> %s: %.2e' % (name, e.max()))
    assert (e <= 1e-5).all(), e
    # and through trafo_adjoint: d<h, A* y>/dy = (A*)^T h = c_w diag(w) J h
    y = torch.randn(B, 1, *geom.obs_shape, device='cuda', generator=gen, requires_grad=True)
    h = torch.rand(B, 1, *geom.im_shape, device='cuda', generator=gen)
    (rt.trafo_adjoint(y) * h).sum().backward()
    ref = M.fp64(og, h.cpu().numpy()) * geom.range_weights[:, None]
    assert (_per_sample(y.grad, ref) <= 1e-5).all()


def test_reference_dps_goldens_on_a_matched_operator(golden, monkeypatch):
    """The reference's DPS goldens (predictors_small.npz) differentiate through torch.sparse, i.e. the exact transpose;
    the matched operator reproduces them to 1e-4 (the pixel-driven one only to the matched/unmatched gap)."""
    from scorenet import BlurScore
    pkg = _pkg()
    d = golden('predictors_small.npz')
    rt = _rt(_geometry('u24'))
    x = torch.from_numpy(d['x']).cuda()
    y = torch.from_numpy(d['y']).cuda()
    nll = lambda v: torch.linalg.norm(y - rt(v))          # noqa: E731
    cpu_randn_like = torch.randn_like
    monkeypatch.setattr(torch, 'randn_like', lambda t, **kw: cpu_randn_like(t.cpu(), **kw).to(t.device))
    errs = {}

    class VpScore(torch.nn.Module):
        def forward(self, v, t):
            return -0.7 * v + 0.1 * torch.tanh(v) * t[:, None, None, None]
    vp, vscore = pkg.VPSDE(), VpScore()
    tv = torch.ones(2, device='cuda') * 0.4
    torch.manual_seed(5)
    a, b = pkg.Euler_Maruyama_sde_predictor(score=vscore, sde=vp, x=x.clone(), time_step=tv, step_size=1e-2,
                                            nloglik=nll, datafitscale=0.4, penalty=0.3, aTweedy=True)
    errs['em_dps_x'], errs['em_dps_mean'] = rel_l2(a.cpu().numpy(), d['em_dps_x']), rel_l2(b.cpu().numpy(), d['em_dps_mean'])
    torch.manual_seed(6)
    out = pkg.Langevin_sde_corrector(score=vscore, sde=vp, x=x.clone(), time_step=tv, nloglik=nll, datafitscale=0.4,
                                     penalty=0.3, corrector_steps=2)
    errs['langevin'] = rel_l2(out.cpu().numpy(), d['langevin'])
    sde, score = pkg.DDPM(), BlurScore().cuda()
    ts = (torch.ones(2, device='cuda') * 400., torch.ones(2, device='cuda') * 390.)
    torch.manual_seed(7)
    a, b = pkg.Ancestral_Sampling(score=score, sde=sde, x=x.clone(), time_step=ts, step_size=1, nloglik=nll, penalty=0.5)
    errs['anc_dps_x'], errs['anc_dps_xhat0'] = rel_l2(a.cpu().numpy(), d['anc_dps_x']), rel_l2(b.cpu().numpy(), d['anc_dps_xhat0'])
    print('\nreference DPS goldens on the matched operator: ' + ', '.join('%s %.2e' % kv for kv in errs.items()))
    for k, e in errs.items():
        assert e <= 1e-4, (k, e)


@pytest.mark.parametrize('dc_type', ['cg', 'gd'])
@pytest.mark.parametrize('batch', [1, 3])
def test_fused_adaptation_objective_on_a_matched_operator(dc_type, batch):
    """scd_adapt_fwd / scd_adapt_bwd against apTweedy -> cg | gradient step -> the loss as a tensor expression,
    differentiated by autograd through trafo / trafo_adjoint."""
    pkg = _pkg()
    from diffusion_models_dev_project_b200.samplers.adaptation import AdaptationLoss, adapt_objective
    for geom in (_G().from_im_shape((64, 64), 23), _G().from_angles((64, 64), AS._golden(23))):
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
        gamma, lam, n_iter = 0.05, 1e-3, 2
        sa = s0.clone().requires_grad_(True)
        la = adapt_objective(sa, x, t, rhs, AdaptationLoss(y, rt, lam), sde, gamma, n_iter, dc_type)
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
        assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-4, (float(la), float(lb))
        assert rel_l2(sa.grad.cpu().numpy(), sb.grad.cpu().numpy()) < 1e-4


# ----------------------------------------------------------------------------------------------- banded ---
@pytest.mark.parametrize('P', [1, 2, 4, 8])
def test_peer_staged_reduction_on_a_matched_operator(P):
    geom = _geometry('u256')
    rt, og = _rt(geom), W.geometry(geom)
    dev = torch.device('cuda')
    n, chunk = 8, 4
    L = E.Layout(geom.im_shape, P, chunk)
    ranges = TB._ranges('u256', rt, P)
    data = _noise((n, 1, *geom.obs_shape), P)
    rt.set_tuning(dev, bp_rows=1)
    n1 = geom.im_shape[1]

    def staged(stage, lo, hi, buf):
        for r in range(P):
            part = rt._bp(data[lo:hi], rt.adj_scale, angle_range=ranges[r])
            for o in range(P):
                row_lo, rows = L.band(o)
                slab = stage[o].view(E.NBUF, P, chunk, L.band_rows, n1)[buf, r, :hi - lo, :rows]
                assert torch.equal(slab, part[:, 0, row_lo:row_lo + rows]), ('slab', lo, r, o)

    result = TB._emulate(rt, L, n, ranges, 'bp', data, staged)
    rt.set_tuning(dev, bp_rows=0)
    e = _per_sample(result[0], M.bp64(og, data.cpu().numpy()))
    print('\nbanded matched P%d: %.2e' % (P, e.max()))
    assert (e <= BP_GATE).all(), e
    for p in range(1, P):
        assert torch.equal(result[p], result[0])


# -------------------------------------------------------------------------------------------------- fbp ---
@pytest.mark.parametrize('name', ['u256', 'wedge90', 'golden37'])
def test_fbp_matches_its_matched_oracle(name):
    geom = _geometry(name)
    rt, og = _rt(geom), W.geometry(geom)
    x = _phantoms(geom.im_shape, 2)
    y = rt(x)
    e = _per_sample(rt.fbp(y), M.fbp64(og, y.cpu().numpy()))
    print('\nfbp matched %s: %.2e' % (name, e.max()))
    assert (e <= 1e-4).all(), e


# ------------------------------------------------------------------------------------------- rejections ---
def test_rejections_write_nothing():
    from diffusion_models_dev_project_b200 import _lib, fused
    lib = _lib.load()
    ang = np.array([0.1, 0.7, 2.0])
    fused.launch_count(reset=True)
    for dx, ds, flags in ((1.5, 1.0, 1), (2.0, 1.0, 1), (1.0, 1.0, 2), (1.0, 1.0, 0x101)):
        d = _lib.GeomDesc(n0=16, n1=16, x_min=-8 * dx, y_min=-8 * dx, dx=dx, n_angles=3,
                          angles=ang.ctypes.data_as(C.POINTER(C.c_double)), n_det=33, s_min=-16.5 * ds, ds=ds,
                          adj_scale=1.0)
        h = C.c_void_p(1)
        assert lib.scd_geom_create_ex(C.byref(d), None, flags, C.byref(h)) == _lib.SCD_E_INVALID, (dx, flags)
        assert not h.value
    assert fused.launch_count() == 0
    # the same geometry at dx/ds = 1.49 is accepted, and the Python layer reports the rejection of an explicit geometry
    d = _lib.GeomDesc(n0=16, n1=16, x_min=-8 * 1.49, y_min=-8 * 1.49, dx=1.49, n_angles=3,
                      angles=ang.ctypes.data_as(C.POINTER(C.c_double)), n_det=33, s_min=-16.5, ds=1.0, adj_scale=1.0)
    h = C.c_void_p()
    assert lib.scd_geom_create_ex(C.byref(d), None, 1, C.byref(h)) == 0 and h.value
    lib.scd_geom_destroy(h)
    G = _G()
    wide = G(n0=16, n1=16, x_min=-16.0, y_min=-16.0, dx=2.0, angles=np.array([0.1, 0.7, 2.0]), n_det=33,
             s_min=-16.5, ds=1.0)
    rt = _pkg().B200RayTrafo((16, 16), 3, geometry=wide, adjoint='matched')
    with pytest.raises(RuntimeError, match='dx/ds < 1.5'):
        rt.trafo_adjoint(torch.zeros(1, 1, 3, 33, device='cuda'))
    assert _pkg().B200RayTrafo((16, 16), 3, geometry=wide)(torch.zeros(1, 1, 16, 16, device='cuda')).shape == (1, 1, 3, 33)
