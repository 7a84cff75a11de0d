"""Generate the golden vectors under tests/golden/ by running the REFERENCE's own code.

Needs a checkout of the reference project, named by SCD_REFERENCE_ROOT:
    SCD_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py

The reference package is imported through oracle/ref_harness.py (third-party imports
stubbed).  Its cg, apTweedy, ddim, DDPM, _schedule_jump, DDS predictor and BaseSampler
run unmodified on CPU; the projector they call is oracle.OracleRayTrafo (sparse Joseph A,
sparse pixel-driven A*), because the reference's own projector (ODL/ASTRA) cannot run here.
"""
import json
import os
import sys
import functools

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import oracle as O          # noqa: E402
from oracle import ref_harness          # noqa: E402
from scorenet import BlurScore          # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
src = ref_harness.import_reference()
from src.utils.cg import cg as ref_cg                                   # noqa: E402
from src.utils.sde import DDPM as RefDDPM                               # noqa: E402
from src.samplers.utils import (ddim as ref_ddim, apTweedy as ref_tweedy, _schedule_jump as ref_jump,  # noqa: E402
                                decomposed_diffusion_sampling_sde_predictor as ref_dds)
from src.samplers.base_sampler import BaseSampler as RefSampler          # noqa: E402
from src.physics.simulation import simulate as ref_simulate             # noqa: E402
from src.utils.metrics import PSNR as ref_psnr                          # noqa: E402

torch.set_num_threads(8)


def schedule_fixture():
    sde = RefDDPM()
    out = {'jump': {}, 'pairs': {}, 'abar': {}, 'mean': {}, 'std': {}}
    for args in [(10, 1, 1), (100, 1, 1), (50, 1, 1), (20, 2, 2), (12, 3, 2)]:
        out['jump']['%d,%d,%d' % args] = ref_jump(*args)
    for n in (10, 50, 100, 1000):
        ts = ref_jump(n, 1, 1)
        skip = sde.num_steps // n
        out['pairs'][str(n)] = [[i * skip, j * skip if j > 0 else -1] for i, j in zip(ts[:-1], ts[1:])]
    t = torch.tensor([-1., 0., 1., 10., 500., 990., 999.])
    ab = sde._compute_alpha_cumprod(t)
    out['abar'] = {'t': t.tolist(), 'bits': ab.numpy().view(np.uint32).tolist()}
    out['mean'] = sde.marginal_prob_mean(t).numpy().view(np.uint32).tolist()
    out['std'] = sde.marginal_prob_std(t).numpy().view(np.uint32).tolist()
    full = sde._compute_alpha_cumprod(torch.arange(-1, 1000).float())
    np.save(os.path.join(OUT, 'abar_table.npy'), full.numpy())
    with open(os.path.join(OUT, 'schedule.json'), 'w') as f:
        json.dump(out, f)


def tweedie_ddim_fixture():
    sde = RefDDPM()
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(3, 1, 16, 20, generator=g)
    s = torch.randn(3, 1, 16, 20, generator=g)
    xhat = torch.randn(3, 1, 16, 20, generator=g)
    res = {'x': x.numpy(), 's': s.numpy(), 'xhat': xhat.numpy()}
    cases = [(990, 980), (500, 490), (20, 10), (10, -1), (0, -1), (300, 310)]
    res['cases'] = np.array(cases)
    for ci, (t, tp) in enumerate(cases):
        tt = torch.ones(3) * t
        tpv = torch.ones(3) * tp
        res['tweedie_%d' % ci] = ref_tweedy(s=s, x=x, sde=sde, time_step=tt).numpy()
        for eta in (0.0, 0.15, 0.85):
            torch.manual_seed(77 + ci)
            out = ref_ddim(sde=sde, s=s, xhat=xhat, time_step=(tt, tpv), step_size=1, eta=eta,
                           use_simplified_eqn=True)
            torch.manual_seed(77 + ci)
            noise = torch.randn_like(xhat)
            res['ddim_%d_%g' % (ci, eta)] = out.numpy()
            res['noise_%d' % ci] = noise.numpy()
    np.savez_compressed(os.path.join(OUT, 'tweedie_ddim.npz'), **res)


def cg_fixture():
    geom = O.OracleGeometry((32, 32), 12)
    rt = O.OracleRayTrafo(geom)
    g = torch.Generator().manual_seed(5)
    x0 = torch.rand(3, 1, 32, 32, generator=g)
    rhs = torch.rand(3, 1, 32, 32, generator=g) * 2
    res = {'x0': x0.numpy(), 'rhs': rhs.numpy(), 'im': np.array([32, 32]), 'num_angles': np.array(12)}
    for gamma in (0.01, 1.0):
        op = lambda v: v + gamma * rt.trafo_adjoint(rt(v))      # noqa: E731
        for k in (0, 1, 2, 5):
            res['x_g%g_k%d' % (gamma, k)] = ref_cg(op=op, x=x0, rhs=rhs, n_iter=k).numpy()
    np.savez_compressed(os.path.join(OUT, 'cg_small.npz'), **res)


def dds_fixture(n_images=2, num_steps=100, cg_iter=5, gamma=0.01, eta=0.15):
    """Config 1 of BASELINE.json: 256x256, 60 angles, B=1, 100 DDIM steps, DDS with CG(5)."""
    phantoms = torch.load(os.path.join(ref_harness.REFERENCE_ROOT, 'dataset', 'disk_ellipses_val_256.pt'))
    geom = O.OracleGeometry((256, 256), 60)
    rt = O.OracleRayTrafo(geom)
    sde = RefDDPM()
    score = BlurScore()
    res = {'num_steps': np.array(num_steps), 'cg_iter': np.array(cg_iter), 'gamma': np.array(gamma),
           'eta': np.array(eta)}
    for i in range(n_images):
        gt = phantoms[i][None]                          # [1,1,256,256]
        torch.manual_seed(1 + i)                        # run_conditional_sampling.py:52-53
        y = ref_simulate(gt, rt, 0.01, rng=np.random.default_rng(1 + i))
        sample_kwargs = {
            'num_steps': num_steps, 'batch_size': 1, 'start_time_step': 0, 'im_shape': [1, 256, 256],
            'eps': 1e-3, 'travel_length': 1, 'travel_repeat': 1,
            'predictor': {'eta': eta, 'gamma': gamma, 'use_simplified_eqn': True, 'ray_trafo': rt}}
        predictor = functools.partial(ref_dds, score=score, sde=sde, rhs=rt.trafo_adjoint(y),
                                      cg_kwargs={'max_iter': cg_iter})
        sampler = RefSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=sample_kwargs,
                             device='cpu')
        recon = sampler.sample(logging=False)
        psnr = ref_psnr(recon[0, 0].numpy(), gt[0, 0].numpy())
        print('image', i, 'PSNR', psnr)
        res['gt_%d' % i] = gt.numpy()
        res['y_%d' % i] = y.numpy()
        res['recon_%d' % i] = recon.numpy()
        res['psnr_%d' % i] = np.array(psnr)
    np.savez_compressed(os.path.join(OUT, 'dds_256.npz'), **res)


def dds_small_fixture():
    """A short chain on a small geometry, batch 2, for fast CPU-side checks of the ports."""
    geom = O.OracleGeometry((64, 64), 16)
    rt = O.OracleRayTrafo(geom)
    sde = RefDDPM()
    score = BlurScore()
    g = torch.Generator().manual_seed(3)
    gt = torch.rand(2, 1, 64, 64, generator=g)
    gt = torch.nn.functional.avg_pool2d(gt, 5, 1, 2)
    y = rt(gt)
    sample_kwargs = {
        'num_steps': 10, 'batch_size': 2, 'start_time_step': 0, 'im_shape': [1, 64, 64],
        'eps': 1e-3, 'travel_length': 1, 'travel_repeat': 1,
        'predictor': {'eta': 0.15, 'gamma': 0.05, 'use_simplified_eqn': True, 'ray_trafo': rt}}
    predictor = functools.partial(ref_dds, score=score, sde=sde, rhs=rt.trafo_adjoint(y),
                                  cg_kwargs={'max_iter': 3})
    sampler = RefSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=sample_kwargs, device='cpu')
    torch.manual_seed(11)
    recon = sampler.sample(logging=False)
    np.savez_compressed(os.path.join(OUT, 'dds_small.npz'), gt=gt.numpy(), y=y.numpy(), recon=recon.numpy())


def predictors_fixture():
    """One step of the other guidance predictors (Euler-Maruyama naive / DPS on a VP schedule, ancestral
    DDPM unconditional / DPS, Langevin corrector), reference code on CPU, oracle operator."""
    from src.samplers.utils import (Euler_Maruyama_sde_predictor as ref_em, Ancestral_Sampling as ref_anc,
                                    Langevin_sde_corrector as ref_lang)
    from src.utils.sde import VPSDE as RefVPSDE
    geom = O.OracleGeometry((24, 24), 8)
    rt = O.OracleRayTrafo(geom)
    g = torch.Generator().manual_seed(21)
    x = torch.randn(2, 1, 24, 24, generator=g)
    gt = torch.rand(2, 1, 24, 24, generator=g)
    y = rt(gt)
    nll = lambda v: torch.linalg.norm(y - rt(v))          # noqa: E731
    score = BlurScore()
    res = {'x': x.numpy(), 'y': y.numpy()}

    class VpScore(torch.nn.Module):                          # score-matching output for a VP schedule
        def forward(self, v, t):
            return -0.7 * v + 0.1 * torch.tanh(v) * t[:, None, None, None]
    vp, vscore = RefVPSDE(), VpScore()
    tv = torch.ones(2) * 0.4
    for name, kw in (('em_plain', {}), ('em_naive', dict(nloglik=nll, datafitscale=0.4, penalty=0.3, aTweedy=False)),
                     ('em_dps', dict(nloglik=nll, datafitscale=0.4, penalty=0.3, aTweedy=True))):
        torch.manual_seed(5)
        a, b = ref_em(score=vscore, sde=vp, x=x.clone(), time_step=tv, step_size=1e-2, **kw)
        res[name + '_x'], res[name + '_mean'] = a.numpy(), b.numpy()
    torch.manual_seed(6)
    res['langevin'] = ref_lang(score=vscore, sde=vp, x=x.clone(), time_step=tv, nloglik=nll, datafitscale=0.4,
                               penalty=0.3, corrector_steps=2).numpy()
    sde = RefDDPM()
    ts = (torch.ones(2) * 400., torch.ones(2) * 390.)
    for name, kw in (('anc_plain', {}), ('anc_dps', dict(nloglik=nll, penalty=0.5))):
        torch.manual_seed(7)
        a, b = ref_anc(score=score, sde=sde, x=x.clone(), time_step=ts, step_size=1, **kw)
        res[name + '_x'], res[name + '_xhat0'] = a.numpy(), b.numpy()
    np.savez_compressed(os.path.join(OUT, 'predictors_small.npz'), **res)


from make_golden_args import adapted_args, adapted_config          # noqa: E402


def adapted_fixture():
    """SCD adapted sampling (BASELINE config 5) through the reference's OWN factory, `_adapt`,
    `adapted_ddim_sde_predictor` and BaseSampler (src/utils/exp_utils.py:225-295,
    src/samplers/utils.py:220-336) on a small geometry; the operator is the oracle with ODL's
    gradient pairing, the score model tests/scorenet.AdaptableScore."""
    from src.utils.exp_utils import get_standard_adapted_sampler as ref_factory
    from scorenet import AdaptableScore
    geom = O.OracleGeometry((48, 48), 12)
    rt = O.OracleRayTrafo(geom, odl_autograd=True)
    g = torch.Generator().manual_seed(9)
    gt = torch.nn.functional.avg_pool2d(torch.rand(2, 1, 48, 48, generator=g), 5, 1, 2)
    y = rt(gt) + 0.01 * torch.randn(2, 1, *geom.obs_shape, generator=g)
    res = {'gt': gt.numpy(), 'y': y.numpy(), 'im': np.array([48, 48]), 'num_angles': np.array(12)}
    for dc in ('cg', 'gd'):
        score = AdaptableScore(r=2, seed=0)
        sampler = ref_factory(adapted_args(dc), adapted_config(2), score, RefDDPM(), rt, observation=y, device='cpu')
        torch.manual_seed(13)
        recon = sampler.sample(logging=False)
        res['recon_' + dc] = recon.numpy()
        for name, prm in score.named_parameters():
            res['param_%s_%s' % (dc, name)] = prm.detach().numpy()
        print('adapted', dc, 'recon norm', float(recon.norm()),
              {n: float(p.detach().norm()) for n, p in score.named_parameters()})
    np.savez_compressed(os.path.join(OUT, 'adapted_small.npz'), **res)


if __name__ == '__main__':
    if sys.argv[1:] == ['adapted']:        # regenerate only the newest fixture
        adapted_fixture()
        sys.exit(0)
    schedule_fixture()
    tweedie_ddim_fixture()
    cg_fixture()
    dds_small_fixture()
    predictors_fixture()
    adapted_fixture()
    dds_fixture()
    print('golden vectors written to', OUT)
