"""GPU parity of the fused CG / Tweedie / DDIM kernels and of the whole DDS sampler against
golden vectors produced by the reference's own code (tests/golden/make_golden.py)."""
import functools

import numpy as np
import pytest
import torch

from conftest import rel_l2
from fp64_reference import cg64
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


def test_tweedie_and_ddim_bit_exact_vs_reference(golden):
    """scd_tweedie_rhs / scd_ddim reproduce the reference's eager fp32 arithmetic bit for bit
    (same inputs, same noise): apTweedy and ddim of reference src/samplers/utils.py."""
    pkg = _pkg()
    from diffusion_models_dev_project_b200 import fused
    d = golden('tweedie_ddim.npz')
    sde = pkg.DDPM()
    abar = sde.alpha_bar_table('cuda')
    x, s, xhat = (torch.from_numpy(d[k]).cuda() for k in ('x', 's', 'xhat'))
    for ci, (t, tp) in enumerate(d['cases']):
        tt = torch.ones(3, device='cuda') * float(t)
        tpv = torch.ones(3, device='cuda') * float(tp)
        tw = fused.tweedie_rhs(x, s, tt, abar).cpu().numpy()
        assert np.array_equal(tw, d['tweedie_%d' % ci]), 'tweedie case %d' % ci
        noise = torch.from_numpy(d['noise_%d' % ci]).cuda()
        for eta in (0.0, 0.15, 0.85):
            out = fused.ddim_ddpm(xhat, s, noise, tt, tpv, abar, eta).cpu().numpy()
            ref = d['ddim_%d_%g' % (ci, eta)]
            assert np.array_equal(out, ref), 'ddim case %d eta %g: max diff %g' % (ci, eta, np.abs(out - ref).max())
    # the public functions route to the same kernels
    tw2 = pkg.apTweedy(s=s, x=x, sde=sde, time_step=torch.ones(3, device='cuda') * 500.)
    assert np.array_equal(tw2.cpu().numpy(), d['tweedie_1'])


def test_tweedie_rhs_fused_b(golden):
    from diffusion_models_dev_project_b200 import fused
    pkg = _pkg()
    d = golden('tweedie_ddim.npz')
    abar = pkg.DDPM().alpha_bar_table('cuda')
    x, s, atb = (torch.from_numpy(d[k]).cuda() for k in ('x', 's', 'xhat'))
    tt = torch.ones(3, device='cuda') * 500.
    xh, b = fused.tweedie_rhs(x, s, tt, abar, atb=atb, gamma=0.01)
    assert np.array_equal(xh.cpu().numpy(), d['tweedie_1'])
    assert torch.equal(b, xh + 0.01 * atb)


@pytest.mark.parametrize('gamma', [0.01, 1.0])
def test_cg_matches_reference_cg(golden, gamma):
    """Fused scd_cg vs the reference's cg() run on the oracle operator (golden), every n_iter.
    Gate 1e-5 rel L2 per iterate; for the ill-conditioned gamma = 1 system fp32 round-off is
    amplified by the recurrences, so there the gate is "no further from the float64 CG iterate
    than the reference's own fp32 result is"."""
    pkg = _pkg()
    d = golden('cg_small.npz')
    geom = O.OracleGeometry((32, 32), 12)
    rt = pkg.B200RayTrafo((32, 32), 12)
    x0 = torch.from_numpy(d['x0']).cuda()
    rhs = torch.from_numpy(d['rhs']).cuda()
    op = rt.normal_op(gamma)
    for k in (0, 1, 2, 5):
        x = pkg.cg(op=op, x=x0, rhs=rhs, n_iter=k).cpu().numpy()
        ref = d['x_g%g_k%d' % (gamma, k)]
        err = rel_l2(x, ref)
        if err >= 1e-5:
            exact = cg64(geom, d['x0'], d['rhs'], gamma, k)
            assert rel_l2(x, exact) <= 4 * rel_l2(ref, exact) + 1e-5, (gamma, k, err, rel_l2(x, exact), rel_l2(ref, exact))
    assert torch.equal(x0, torch.from_numpy(d['x0']).cuda())        # start value untouched


def test_cg_generic_path_equals_fused_path():
    """cg() with a plain closure (tensor-op recurrences, CUDA A/A*) and the fused solve agree."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((96, 96), 18)
    gen = torch.Generator(device='cuda').manual_seed(1)
    x0 = torch.rand(4, 1, 96, 96, device='cuda', generator=gen)
    rhs = torch.rand(4, 1, 96, 96, device='cuda', generator=gen)
    fusedx = pkg.cg(op=rt.normal_op(0.05), x=x0, rhs=rhs, n_iter=4)
    plain = pkg.cg(op=lambda v: v + 0.05 * rt.trafo_adjoint(rt(v)), x=x0, rhs=rhs, n_iter=4)
    # two fp32 evaluations of the same recurrences (fma vs mul+add, different reduction trees)
    assert rel_l2(fusedx.cpu().numpy(), plain.cpu().numpy()) < 1e-4


def test_cg_converges_on_full_size_batch():
    """Size-independent property at the bench size: residual of (I + gamma A*A) x = b drops."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((256, 256), 60)
    gen = torch.Generator(device='cuda').manual_seed(2)
    x0 = torch.rand(8, 1, 256, 256, device='cuda', generator=gen)
    b = torch.rand(8, 1, 256, 256, device='cuda', generator=gen) * 3
    op = rt.normal_op(0.01)
    r0 = (b - op(x0)).flatten(1).norm(dim=1)
    prev = r0
    for k in (1, 5, 20):
        x = pkg.cg(op=op, x=x0, rhs=b, n_iter=k)
        r = (b - op(x)).flatten(1).norm(dim=1)
        assert bool((r < prev).all()), (k, r, prev)
        prev = r
    assert float((prev / r0).max()) < 1e-2


def _patch_noise_to_cpu_generator(monkeypatch):
    """The golden chains were produced on CPU, where randn_like draws from the CPU generator."""
    real = torch.randn_like

    def cpu_randn_like(t, **kw):
        return torch.randn(t.shape, dtype=t.dtype).to(t.device)
    monkeypatch.setattr(torch, 'randn_like', cpu_randn_like)
    return real


def test_dds_small_chain_matches_reference(golden, monkeypatch):
    pkg = _pkg()
    from scorenet import BlurScore
    _patch_noise_to_cpu_generator(monkeypatch)
    d = golden('dds_small.npz')
    rt = pkg.B200RayTrafo((64, 64), 16)
    sde = pkg.DDPM()
    score = BlurScore().cuda()
    y = torch.from_numpy(d['y']).cuda()
    kw = {'num_steps': 10, 'batch_size': 2, 'start_time_step': 0, 'im_shape': [1, 64, 64], 'eps': 1e-3,
          'travel_length': 1, 'travel_repeat': 1,
          'predictor': {'eta': 0.15, 'gamma': 0.05, 'use_simplified_eqn': True, 'ray_trafo': rt}}
    predictor = functools.partial(pkg.decomposed_diffusion_sampling_sde_predictor, score=score, sde=sde,
                                  rhs=rt.trafo_adjoint(y), cg_kwargs={'max_iter': 3})
    sampler = pkg.BaseSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=kw, device='cuda')
    torch.manual_seed(11)
    recon = sampler.sample(logging=False).cpu().numpy()
    assert rel_l2(recon, d['recon']) < 1e-4


def test_cg_gradient_fused_reverse_sweep_equals_autograd():
    """Differentiating `cg` on the CUDA operator: the hand-written reverse sweep (no autograd graph, A*A through
    the fused kernels) against autograd through the tensor recurrences with the A / A* autograd Functions."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((64, 64), 16)
    gamma = 0.05
    op = rt.normal_op(gamma)
    generic = lambda v: v + gamma * rt.trafo_adjoint(rt(v))          # noqa: E731  (plain callable: tensor path)
    gen = torch.Generator(device='cuda').manual_seed(0)
    for k in (1, 3):
        x = torch.rand(3, 1, 64, 64, device='cuda', generator=gen, requires_grad=True)
        b = (torch.rand(3, 1, 64, 64, device='cuda', generator=gen) + 1.0).requires_grad_()
        w = torch.randn(3, 1, 64, 64, device='cuda', generator=gen)
        out = pkg.cg(op, x, b, k)
        assert out.grad_fn is not None and 'CgSelfAdjoint' in type(out.grad_fn).__name__
        gx, gb = torch.autograd.grad((out * w).sum(), (x, b))
        ref = pkg.cg(generic, x, b, k)
        gx_ref, gb_ref = torch.autograd.grad((ref * w).sum(), (x, b))
        assert rel_l2(out.detach().cpu().numpy(), ref.detach().cpu().numpy()) < 1e-5
        assert rel_l2(gx.cpu().numpy(), gx_ref.cpu().numpy()) < 1e-4, k
        assert rel_l2(gb.cpu().numpy(), gb_ref.cpu().numpy()) < 1e-4, k


@pytest.mark.parametrize('cuda_graph', [False, True])
def test_adapted_sampling_matches_reference_chain(golden, monkeypatch, cuda_graph):
    """(cuda_graph: the Adam step -- score model, scd_adapt_fwd / scd_adapt_bwd, optimizer -- captured once and
    replayed, samplers/utils.py:_AdaptGraph.)
    BASELINE config 5 (SCD adapted sampling): factory -> `_adapt` (Adam through Tweedie, CG, A, A* and
    the fused adaptation loss) -> adapted predictor -> sampler on the CUDA kernels, against the outputs
    of the reference's own get_standard_adapted_sampler / _adapt / adapted_ddim_sde_predictor /
    BaseSampler (tests/golden/make_golden.py:adapted_fixture; operator = oracle with ODL's gradient
    pairing).  Checks the reconstruction and the adapted parameters, for dc_type cg and gd."""
    pkg = _pkg()
    from make_golden_args import adapted_args, adapted_config
    from scorenet import AdaptableScore
    from diffusion_models_dev_project_b200.utils import exp_utils as E
    _patch_noise_to_cpu_generator(monkeypatch)
    d = golden('adapted_small.npz')
    rt = pkg.B200RayTrafo(tuple(int(v) for v in d['im']), int(d['num_angles']))
    y = torch.from_numpy(d['y']).cuda()
    for dc in ('cg', 'gd'):
        score = AdaptableScore(r=2, seed=0).cuda()
        args = adapted_args(dc)
        args.adapt_cuda_graph = cuda_graph
        sampler = E.get_standard_adapted_sampler(args, adapted_config(2, 'cuda'), score, pkg.DDPM(), rt,
                                                 observation=y, device='cuda')
        torch.manual_seed(13)
        recon = sampler.sample(logging=False).cpu().numpy()
        assert rel_l2(recon, d['recon_' + dc]) < 1e-4, (dc, rel_l2(recon, d['recon_' + dc]))
        for name, prm in score.named_parameters():
            ref = d['param_%s_%s' % (dc, name)]
            assert np.allclose(prm.detach().cpu().numpy(), ref, atol=2e-5), (dc, name, prm, ref)
        assert score.adapter.scale == 1.0
        assert (getattr(score, '_scd_adapt_graph', None) is not None) == cuda_graph


def test_dds_256_reconstruction_psnr_parity(golden, monkeypatch):
    """BASELINE config 1: 256x256, 60 angles, B=1, 100 DDIM steps, CG(5), gamma 0.01, eta 0.15.
    Gate: PSNR within 0.1 dB of the reference sampler (same seeds)."""
    pkg = _pkg()
    from scorenet import BlurScore
    _patch_noise_to_cpu_generator(monkeypatch)
    d = golden('dds_256.npz')
    rt = pkg.B200RayTrafo((256, 256), 60)
    sde = pkg.DDPM()
    score = BlurScore().cuda()
    for i in range(2):
        gt = d['gt_%d' % i]
        y = torch.from_numpy(d['y_%d' % i]).cuda()
        kw = {'num_steps': int(d['num_steps']), 'batch_size': 1, 'start_time_step': 0, 'im_shape': [1, 256, 256],
              'eps': 1e-3, 'travel_length': 1, 'travel_repeat': 1,
              'predictor': {'eta': float(d['eta']), 'gamma': float(d['gamma']), 'use_simplified_eqn': True,
                            'ray_trafo': rt}}
        predictor = functools.partial(pkg.decomposed_diffusion_sampling_sde_predictor, score=score, sde=sde,
                                      rhs=rt.trafo_adjoint(y), cg_kwargs={'max_iter': int(d['cg_iter'])})
        sampler = pkg.BaseSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=kw, device='cuda')
        torch.manual_seed(1 + i)
        recon = sampler.sample(logging=False).cpu().numpy()
        psnr = pkg.PSNR(recon[0, 0], gt[0, 0])
        assert abs(psnr - float(d['psnr_%d' % i])) < 0.1, (psnr, float(d['psnr_%d' % i]))
        assert rel_l2(recon, d['recon_%d' % i]) < 1e-3


def test_autograd_pairing_matches_odl_convention():
    """grad through trafo = A*(g)/c_w, through trafo_adjoint = c_w*A(g) (SURVEY.md section 8b), and the
    differentiable cg (SCD adaptation path) backpropagates."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((64, 64), 12)
    c_w = rt.geometry.range_weight
    gen = torch.Generator(device='cuda').manual_seed(3)
    x = torch.rand(2, 1, 64, 64, device='cuda', generator=gen, requires_grad=True)
    g = torch.randn(2, 1, *rt.obs_shape, device='cuda', generator=gen)
    (rt(x) * g).sum().backward()
    assert rel_l2(x.grad.cpu().numpy(), (rt.trafo_adjoint(g) / c_w).cpu().numpy()) < 1e-6
    y = torch.randn(2, 1, *rt.obs_shape, device='cuda', generator=gen, requires_grad=True)
    h = torch.rand(2, 1, 64, 64, device='cuda', generator=gen)
    (rt.trafo_adjoint(y) * h).sum().backward()
    assert rel_l2(y.grad.cpu().numpy(), (c_w * rt(h)).cpu().numpy()) < 1e-6
    # gradient through the CG recurrences w.r.t. the start value / rhs
    x0 = torch.rand(2, 1, 64, 64, device='cuda', generator=gen, requires_grad=True)
    out = pkg.cg(op=rt.normal_op(0.1), x=x0, rhs=x0 + 0.1 * h, n_iter=2)
    out.square().sum().backward()
    assert torch.isfinite(x0.grad).all() and float(x0.grad.abs().max()) > 0


def test_adaptation_loss_fused_matches_tensor_expression():
    """mean((Ax-y)^2) + lam*tv(x): fused kernels with hand-written backward vs the reference's tensor
    expression differentiated by autograd (reference src/utils/exp_utils.py:256-257, adaptation.py:7-11)."""
    pkg = _pkg()
    for shape, na, batch in (((64, 64), 12, 2), ((48, 80), 7, 1), ((256, 256), 60, 1)):
        rt = pkg.B200RayTrafo(shape, na)
        gen = torch.Generator(device='cuda').manual_seed(5)
        x = torch.rand(batch, 1, *shape, device='cuda', generator=gen)
        x[..., 3:9, 5:11] = 0.5                                   # flat patch: sign(0) = 0 in the TV gradient
        y = rt(torch.rand(1, 1, *shape, device='cuda', generator=gen))
        lam = 1e-3
        xa = x.clone().requires_grad_(True)
        la = pkg.adaptation_loss(xa, y, rt, lam)
        (3.0 * la).backward()
        xb = x.clone().requires_grad_(True)
        lb = torch.mean((rt(xb) - y).pow(2)) + lam * pkg.tv_loss(xb)
        (3.0 * lb).backward()
        assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-5
        assert rel_l2(xa.grad.cpu().numpy(), xb.grad.cpu().numpy()) < 1e-5


def test_dps_predictors_differentiate_through_the_cuda_projector(golden, monkeypatch):
    """DPS (ancestral, DDPM) and Euler-Maruyama DPS (VP) on the GPU: the data-fit gradient flows through
    fp_march / bp_tile via the autograd Functions.  The CPU golden uses the exact transpose of A in the
    backward, the ODL pairing uses the pixel-driven A*/c_w: agreement to the matched/unmatched gap."""
    from scorenet import BlurScore
    pkg = _pkg()
    d = golden('predictors_small.npz')
    rt = pkg.B200RayTrafo((24, 24), 8)
    x = torch.from_numpy(d['x']).cuda()
    y = torch.from_numpy(d['y']).cuda()
    nll = lambda v: torch.linalg.norm(y - rt(v))          # noqa: E731
    torch.manual_seed(7)
    noise = torch.randn(2, 1, 24, 24)
    monkeypatch.setattr(torch, 'randn_like', lambda t: noise.to(t.device))
    sde, score = pkg.DDPM(), BlurScore().cuda()
    ts = (torch.ones(2, device='cuda') * 400., torch.ones(2, device='cuda') * 390.)
    a, b = pkg.Ancestral_Sampling(score=score, sde=sde, x=x.clone(), time_step=ts, step_size=1, nloglik=nll, penalty=0.5)
    assert rel_l2(b.cpu().numpy(), d['anc_dps_xhat0']) < 1e-5
    assert rel_l2(a.cpu().numpy(), d['anc_dps_x']) < 2e-2
    a0, _ = pkg.Ancestral_Sampling(score=score, sde=sde, x=x.clone(), time_step=ts, step_size=1)
    assert rel_l2(a0.cpu().numpy(), d['anc_plain_x']) < 1e-5
    assert float((a - a0).abs().max()) > 0                    # the guidance term acted


def test_bitwise_reproducible_across_runs():
    """No atomics anywhere on the path: partial sums are added in a fixed order (cluster ranks, per-CTA
    partials), so repeated calls return bit-identical tensors."""
    pkg = _pkg()
    dev = torch.device('cuda')
    for shape, na, B in (((256, 256), 60, 8), ((96, 80), 18, 3), ((256, 256), 60, 40)):
        rt = pkg.B200RayTrafo(shape, na)
        gen = torch.Generator(device=dev).manual_seed(13)
        x = torch.rand(B, 1, *shape, device=dev, generator=gen)
        s = torch.randn(B, 1, *shape, device=dev, generator=gen)
        eps = torch.randn(B, 1, *shape, device=dev, generator=gen)
        abar = pkg.DDPM().alpha_bar_table(dev)
        t = torch.ones(B, device=dev) * 300.
        tp = torch.ones(B, device=dev) * 290.
        y = rt(x)
        atb = rt.trafo_adjoint(y)
        first = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
        for _ in range(3):
            assert torch.equal(rt(x), y) and torch.equal(rt.trafo_adjoint(y), atb)
            again = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
            assert torch.equal(again[0], first[0]) and torch.equal(again[1], first[1])


def test_dds_step_is_cuda_graph_capturable():
    """The library never allocates or synchronises: a whole data-consistency step (24 launches with
    programmatic dependent launch) captures into a CUDA graph and replays with new inputs."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((96, 96), 20)
    dev = torch.device('cuda')
    gen = torch.Generator(device=dev).manual_seed(8)
    B = 4
    abar = pkg.DDPM().alpha_bar_table(dev)
    x = torch.rand(B, 1, 96, 96, device=dev, generator=gen)
    s = torch.randn(B, 1, 96, 96, device=dev, generator=gen)
    eps = torch.randn(B, 1, 96, 96, device=dev, generator=gen)
    atb = rt.trafo_adjoint(rt(torch.rand(B, 1, 96, 96, device=dev, generator=gen)))
    t = torch.ones(B, device=dev) * 700.
    tp = torch.ones(B, device=dev) * 690.
    rt.dds_step(x, s, atb, eps, t, tp, abar, 0.05, 0.15, 3)               # warm-up: handles, workspace
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, xh = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.05, 0.15, 3)
    for k in range(2):
        x.copy_(torch.rand(B, 1, 96, 96, device=dev, generator=gen))
        s.copy_(torch.randn(B, 1, 96, 96, device=dev, generator=gen))
        t.fill_(500. - 100 * k); tp.fill_(490. - 100 * k)
        graph.replay()
        ref, refh = rt.dds_step(x, s, atb, eps, t, tp, abar, 0.05, 0.15, 3)
        assert torch.equal(out, ref) and torch.equal(xh, refh)


def test_fbp_inverts_dense_view_projection():
    pkg = _pkg()
    rt = pkg.B200RayTrafo((128, 128), 360)
    k = np.arange(128) - 64 + 0.5
    img = ((k[:, None] / 40) ** 2 + (k[None, :] / 25) ** 2 <= 1).astype(np.float32)
    img += 0.5 * (((k[:, None] - 10) ** 2 + (k[None, :] + 5) ** 2) <= 100)
    x = torch.from_numpy(img)[None, None].cuda()
    rec = rt.fbp(rt(x))
    assert pkg.PSNR(rec[0, 0].cpu().numpy(), img) > 22.0
    assert abs(float(rec.mean() / x.mean()) - 1) < 0.05


def test_workspace_validation():
    import ctypes as C
    from diffusion_models_dev_project_b200 import _lib
    pkg = _pkg()
    rt = pkg.B200RayTrafo((32, 32), 6)
    h = rt._handle(torch.device('cuda'))
    x = torch.rand(1, 1, 32, 32, device='cuda')
    w = torch.empty(1024, dtype=torch.uint8, device='cuda')
    rc = h._lib.scd_cg(h.ptr, x.data_ptr(), x.data_ptr(), 0.1, 1, 1, w.data_ptr(), 1024, None)
    assert rc == _lib.SCD_E_WORKSPACE
    assert int(h._lib.scd_cg_workspace_bytes(h.ptr, 1)) > 5 * 32 * 32 * 4


@pytest.mark.parametrize('dc_type,n_iter', [('cg', 1), ('cg', 3), ('cg', 0), ('dc', 1), ('none', 1)])
@pytest.mark.parametrize('batch', [1, 2, 5])
def test_fused_adaptation_objective_matches_the_tensor_path(dc_type, n_iter, batch):
    """scd_adapt_fwd / scd_adapt_bwd (Tweedie -> CG | gradient step | none -> loss, and the hand-written reverse
    sweep) against the tensor path: apTweedy, the differentiable cg, adaptation_loss, differentiated by autograd --
    what `_adapt` evaluates per Adam step (reference src/samplers/utils.py:241-260)."""
    pkg = _pkg()
    from diffusion_models_dev_project_b200.samplers.adaptation import AdaptationLoss, adapt_objective
    rt = pkg.B200RayTrafo((64, 64), 16)
    sde = pkg.DDPM()
    gen = torch.Generator(device='cuda').manual_seed(17)
    gt = torch.rand(batch, 1, 64, 64, device='cuda', generator=gen)
    gt = torch.nn.functional.avg_pool2d(gt, 5, 1, 2)
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
    assert la is not None and la.dim() == 0
    (3.0 * la).backward()

    sb = s0.clone().requires_grad_(True)
    xhat0 = pkg.apTweedy(s=sb, x=x, sde=sde, time_step=t)
    if dc_type == 'cg':
        xhat = pkg.cg(op=rt.normal_op(gamma), x=xhat0, rhs=xhat0 + gamma * rhs, n_iter=n_iter)
    elif dc_type == 'dc':
        xhat = xhat0 - gamma * rt.trafo_adjoint(rt(xhat0)) + gamma * rhs
    else:
        xhat = xhat0
    lb = loss_fn(x=xhat)
    (3.0 * lb).backward()
    assert abs(float(la) - float(lb)) / abs(float(lb)) < 1e-5, (float(la), float(lb))
    assert rel_l2(sa.grad.cpu().numpy(), sb.grad.cpu().numpy()) < 1e-4
    # the saved state is released by the first backward pass: a second one is refused, not a use-after-free
    if batch == 1 and dc_type == 'cg' and n_iter == 1:
        sc = s0.clone().requires_grad_(True)
        lc = adapt_objective(sc, x, t, rhs, loss_fn, sde, gamma, n_iter, dc_type)
        lc.backward(retain_graph=True)
        with pytest.raises(RuntimeError, match='already differentiated'):
            lc.backward()
    # no fused path for other losses / operators: the caller falls back to the tensor expression
    assert adapt_objective(sa, x, t, rhs, lambda x: x.sum(), sde, gamma, n_iter, dc_type) is None
