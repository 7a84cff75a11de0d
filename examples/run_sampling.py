#!/usr/bin/env python
"""Synthetic-data counterpart of the reference's run_conditional_sampling.py / run_adapted_sampling.py.

Same argument names and the same factory calls (`get_standard_sde`, `get_standard_ray_trafo`,
`get_data_from_ground_truth`, `get_standard_sampler` / `get_standard_adapted_sampler`), with what the
offline container cannot provide replaced by synthetic stand-ins: disk-ellipse phantoms instead of the
datasets, a randomly initialised ADM UNet instead of a checkpoint (so the PSNR it prints measures the
data-consistency path, not a trained prior), a small LoRA injector instead of the vendored one.

    python examples/run_sampling.py --mode conditional --method dds --num_steps 20
    python examples/run_sampling.py --mode adapted --num_steps 10 --num_optim_step 2 --add_cg
    python examples/run_sampling.py --num_steps 20 --angle_range 0 90        # limited angle: a 90 degree wedge
    python examples/run_sampling.py --num_steps 20 --angles_file views.txt   # sparse / non-uniform views
"""
import argparse
import os
import sys
from types import SimpleNamespace as NS

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import diffusion_models_dev_project_b200 as pkg                      # noqa: E402
from bench_support.adm_unet import small_unet, aapm_unet            # noqa: E402
from bench_support.phantoms import disk_ellipses                    # noqa: E402
from bench_support.lora import inject_trainable_lora                # noqa: E402


def parse():
    p = argparse.ArgumentParser(description='conditional / adapted sampling on synthetic data')
    p.add_argument('--mode', default='conditional', choices=['conditional', 'adapted'])
    p.add_argument('--method', default='dds', choices=['naive', 'dps', 'dds'])
    p.add_argument('--sde', default='ddpm', choices=['vpsde', 'vesde', 'ddpm'])
    p.add_argument('--num_steps', default=100)
    p.add_argument('--penalty', default=1)
    p.add_argument('--gamma', default=0.01)
    p.add_argument('--eta', default=0.15)
    p.add_argument('--cg_iter', default=5)
    p.add_argument('--pct_chain_elapsed', default=0)
    p.add_argument('--noise_level', default=0.01)
    p.add_argument('--early_stopping_pct', default=1.0)
    # adapted sampling (run_adapted_sampling.py)
    p.add_argument('--adaptation', default='lora', choices=['lora', 'decoder', 'full'])
    p.add_argument('--num_optim_step', default=10)
    p.add_argument('--adapt_freq', default=1)
    p.add_argument('--lora_include_blocks', default=None, nargs='+')
    p.add_argument('--lora_rank', default=4)
    p.add_argument('--lr', default=1e-3)
    p.add_argument('--tv_penalty', default=1e-6)
    p.add_argument('--add_cg', action='store_true')
    p.add_argument('--dc_type', default='cg', choices=['cg', 'gd', 'none'])
    p.add_argument('--adapt_cuda_graph', action='store_true',
                   help='adapted mode: capture one Adam step (score model, scd_adapt_fwd / scd_adapt_bwd, optimizer) in a '
                        'CUDA graph and replay it')
    # synthetic set-up
    p.add_argument('--im_size', type=int, default=256)
    p.add_argument('--num_angles', type=int, default=60)
    p.add_argument('--angle_range', type=float, nargs=2, default=None, metavar=('MIN', 'MAX'),
                   help='limited angle: num_angles cell-centred views on [MIN, MAX) degrees instead of [0, 180)')
    p.add_argument('--angles_file', default=None,
                   help='text file of view angles in degrees (whitespace or newline separated), weighted by their '
                        'angular cells; replaces --num_angles')
    p.add_argument('--batch_size', type=int, default=1)
    p.add_argument('--num_images', type=int, default=1)
    p.add_argument('--unet', default='small', choices=['small', 'aapm', 'blur'],
                   help="score model: random-init ADM UNet, or 'blur' = the weight-free plug-and-play denoiser of "
                        "tests/scorenet.py (DDPM only; gives a meaningful PSNR without a checkpoint)")
    p.add_argument('--seed', type=int, default=1)
    return p.parse_args()


def main():
    args = parse()
    device = torch.device('cuda')
    forward_op = NS(trafo_name='simple_trafo', num_angles=args.num_angles, impl='b200')
    if args.angle_range is not None and args.angles_file is not None:
        raise SystemExit('give --angle_range or --angles_file, not both')
    if args.angle_range is not None:
        forward_op.angle_range = tuple(np.deg2rad(args.angle_range))
    if args.angles_file is not None:
        forward_op.angles = np.deg2rad(np.loadtxt(args.angles_file, dtype=np.float64).reshape(-1))
        forward_op.num_angles = int(forward_op.angles.size)
    config = NS(
        device=device, seed=args.seed,
        sde=NS(type=args.sde, beta_min=1e-4, beta_max=0.02, num_steps=1000, sigma_min=0.01, sigma_max=50.),
        data=NS(im_size=args.im_size, stddev=float(args.noise_level)),
        forward_op=forward_op,
        sampling=NS(batch_size=args.batch_size, eps=1e-3, travel_length=1, travel_repeat=1),
        model=NS(in_channels=1))
    if args.sde != 'ddpm':
        config.sde.beta_min, config.sde.beta_max = 0.1, 20.
    torch.manual_seed(config.seed)
    sde = pkg.get_standard_sde(config=config)
    torch.manual_seed(0)
    if args.unet == 'blur':
        sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests'))
        from scorenet import BlurScore
        score = BlurScore().to(device).eval()
    else:
        score = (small_unet() if args.unet == 'small' else aapm_unet()).to(device).eval()
    ray_trafo = pkg.get_standard_ray_trafo(config=config).to(device=device)
    phantoms = torch.from_numpy(disk_ellipses(args.num_images, args.im_size, seed=1))
    psnrs = []
    for i in range(args.num_images):
        ground_truth = phantoms[i:i + 1].to(device).expand(args.batch_size, -1, -1, -1).contiguous()
        torch.manual_seed(config.seed + i)
        np.random.seed(config.seed + i)
        _, observation, filtbackproj = pkg.get_data_from_ground_truth(
            ground_truth=ground_truth, ray_trafo=ray_trafo, white_noise_rel_stddev=config.data.stddev)
        if args.mode == 'conditional':
            sampler = pkg.get_standard_sampler(args=args, config=config, score=score, sde=sde, ray_trafo=ray_trafo,
                                               observation=observation, filtbackproj=filtbackproj, device=device)
        else:
            args.method = 'dds'
            import copy
            sampler = pkg.get_standard_adapted_sampler(args=args, config=config, score=copy.deepcopy(score), sde=sde,
                                                       ray_trafo=ray_trafo, observation=observation, device=device,
                                                       lora_inject_fn=inject_trainable_lora)
        recon = sampler.sample(logging=False)
        psnr = pkg.PSNR(recon[0, 0].cpu().numpy(), ground_truth[0, 0].cpu().numpy())
        psnr_fbp = pkg.PSNR(filtbackproj[0, 0].cpu().numpy(), ground_truth[0, 0].cpu().numpy())
        print('image %d: PSNR %.2f dB (FBP %.2f dB)' % (i, psnr, psnr_fbp))
        psnrs.append(psnr)
    print('mean PSNR %.2f dB over %d image(s)' % (float(np.mean(psnrs)), len(psnrs)))


if __name__ == '__main__':
    main()
