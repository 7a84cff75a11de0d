"""Golden fixture of BASELINE config 1 as SURVEY.md section 8(d) specifies it: all 10 vendored disk-ellipse
phantoms (reference dataset/disk_ellipses_val_256.pt), 256x256, 60 angles, conditional DDS sampling at batch 1,
100 DDIM steps, CG(5), gamma 0.01, eta 0.15 (reference run_conditional_sampling.py:20-24), seeds
torch.manual_seed(1 + i) per image (:52-53), relative noise 0.01 from a seeded numpy generator, and the small
ADM UNet of section 8(d) as score model (bench_support.adm_unet.small_unet, torch.manual_seed(0) construction,
random init -- the same weights are rebuilt on the GPU side).

The chain is the REFERENCE's own code: src.samplers.base_sampler.BaseSampler driving
src.samplers.utils.decomposed_diffusion_sampling_sde_predictor (which calls the reference's apTweedy, cg, ddim)
on CPU.  The projector it calls is the C oracle (oracle/ray_oracle.c) behind a small torch adapter, because the
reference's own projector (ODL/ASTRA) cannot run here.

    SCD_REFERENCE_ROOT=<checkout> python tests/golden/make_golden_config1.py    # ~10 min on 8 cores; writes tests/golden/config1_256.npz

Stored per image i: gt_i (fp32), y_i (noisy sinogram made by the reference's `simulate`), fbp-free;
psnr_i of the reference reconstruction; recon_i in full for i < 3 and as 4x4 block means for all i.
"""
import functools
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import oracle as O          # noqa: E402
from oracle import ref_harness          # noqa: E402
from bench_support.adm_unet import small_unet      # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
src = ref_harness.import_reference()
from src.utils.sde import DDPM as RefDDPM                               # noqa: E402
from src.samplers.utils import decomposed_diffusion_sampling_sde_predictor as ref_dds      # noqa: E402
from src.samplers.base_sampler import BaseSampler as RefSampler          # noqa: E402
from src.physics.simulation import simulate as ref_simulate             # noqa: E402
from src.utils.metrics import PSNR as ref_psnr                          # noqa: E402

torch.set_num_threads(8)


class COracleTrafo:
    """torch adapter of the C oracle (A = oracle_fp, A* = oracle_bp)."""

    def __init__(self, geom):
        self.geom = geom
        self.im_shape, self.obs_shape = geom.im_shape, geom.obs_shape

    def trafo(self, x):
        return torch.from_numpy(O.fp(self.geom, x.detach().numpy()))

    def trafo_adjoint(self, y):
        return torch.from_numpy(O.bp(self.geom, y.detach().numpy()))

    __call__ = trafo


def block_means(a, k=4):
    n0, n1 = a.shape[-2:]
    return a.reshape(*a.shape[:-2], n0 // k, k, n1 // k, k).mean(axis=(-3, -1))


def main(num_steps=100, cg_iter=5, gamma=0.01, eta=0.15, n_images=10):
    phantoms = torch.load(os.path.join(ref_harness.REFERENCE_ROOT, 'dataset', 'disk_ellipses_val_256.pt'))
    geom = O.OracleGeometry((256, 256), 60)
    rt = COracleTrafo(geom)
    sde = RefDDPM()
    torch.manual_seed(0)
    score = small_unet().eval()
    res = {'num_steps': np.array(num_steps), 'cg_iter': np.array(cg_iter), 'gamma': np.array(gamma),
           'eta': np.array(eta), 'n_images': np.array(n_images)}
    for i in range(n_images):
        gt = phantoms[i][None].float()                    # [1,1,256,256]
        torch.manual_seed(1 + i)                          # run_conditional_sampling.py:52-53
        y = ref_simulate(gt, rt, 0.01, rng=np.random.default_rng(1 + i))
        kw = {'num_steps': num_steps, 'batch_size': 1, 'start_time_step': 0, 'im_shape': [1, 256, 256],
              'eps': 1e-3, 'travel_length': 1, 'travel_repeat': 1,
              'predictor': {'eta': eta, 'gamma': gamma, 'use_simplified_eqn': True, 'ray_trafo': rt}}
        predictor = functools.partial(ref_dds, score=score, sde=sde, rhs=rt.trafo_adjoint(y),
                                      cg_kwargs={'max_iter': cg_iter})
        sampler = RefSampler(score=score, sde=sde, predictor=predictor, sample_kwargs=kw, device='cpu')
        recon = sampler.sample(logging=False)
        psnr = ref_psnr(recon[0, 0].numpy(), gt[0, 0].numpy())
        print('image', i, 'PSNR', psnr, flush=True)
        res['gt_%d' % i] = gt.numpy()
        res['y_%d' % i] = y.numpy()
        res['psnr_%d' % i] = np.array(psnr)
        res['recon_blk_%d' % i] = block_means(recon.numpy())
        if i < 3:
            res['recon_%d' % i] = recon.numpy()
    np.savez_compressed(os.path.join(OUT, 'config1_256.npz'), **res)
    print('written', os.path.join(OUT, 'config1_256.npz'))


if __name__ == '__main__':
    main()
