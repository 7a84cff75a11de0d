"""Cost of view weights: the fused DDS step (scd_dds_step, CG(5)) on weighted and unweighted geometries.

    python tools/angle_set_bench.py [--reps 7] [--iters 50] [--out FILE]

Gate pair (256 x 256, 60 views, batches 8 and 256): the default geometry (60 views on [0, pi), no weight table)
against a weighted 60-view set (60 of 180 uniform views kept at random: cells from 0.3x to 3x the mean).  A
weighted geometry adds one multiply per ray output of the projector's interleaved sinogram and none to the
backprojector's march, so the two should time the same.  The two geometries are timed alternately, `--reps`
rounds of `--iters` steps each (CUDA events around the round), so that drift of the shared machine hits both;
the JSON gives the median and the spread (min, max) of the rounds.  For information, the step time on sparse
sets of 1-8 views and on a 90 degree wedge: few views give the projector few work units, so these are latency
figures.  The card's name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
from math import pi

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import diffusion_models_dev_project_b200 as pkg                                   # noqa: E402
from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D as G    # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = 'unknown'
    return {'name': name, 'power_limit_and_max_sm_clock': out}


def make_step(geom, batch, seed=0):
    rt = pkg.B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom)
    gen = torch.Generator(device='cuda').manual_seed(seed)
    x, s, eps = (torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen) for _ in range(3))
    atb = rt.trafo_adjoint(rt(torch.rand(batch, 1, *geom.im_shape, device='cuda', generator=gen)))
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t = torch.full((batch,), 500., device='cuda')
    tp = torch.full((batch,), 490., device='cuda')

    def step():
        return rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)
    return step


def time_round(step, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        out = step()
    b.record()
    torch.cuda.synchronize()
    assert torch.isfinite(out[0]).all()
    return a.elapsed_time(b) * 1e3 / iters                 # us per step


def alternate(steps, reps, iters):
    for st in steps.values():                             # warm-up: module load, plans, workspaces
        for _ in range(5):
            st()
    torch.cuda.synchronize()
    times = {k: [] for k in steps}
    for _ in range(reps):
        for k, st in steps.items():
            times[k].append(time_round(st, iters))
    return {k: {'median_us': float(np.median(v)), 'min_us': float(np.min(v)), 'max_us': float(np.max(v)),
                'rounds': len(v)} for k, v in times.items()}


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--reps', type=int, default=7)
    p.add_argument('--iters', type=int, default=50)
    p.add_argument('--out', default=None, help='also write the JSON here')
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('angle_set_bench needs a CUDA device')
    shape = (256, 256)
    keep = np.sort(np.random.default_rng(2024).choice(180, 60, replace=False))
    weighted = G.from_angles(shape, (keep + 0.5) * (pi / 180))
    assert weighted.angle_weights is not None
    res = {'card': card(), 'step': 'dds_step CG(5), gamma 0.01, eta 0.15', 'shape': list(shape), 'gate': {}, 'info': {}}
    for batch in (8, 256):
        steps = {'default_60': make_step(G.from_im_shape(shape, 60), batch),
                 'weighted_60_random_gaps': make_step(weighted, batch)}
        r = alternate(steps, a.reps, a.iters)
        r['weighted_over_default'] = r['weighted_60_random_gaps']['median_us'] / r['default_60']['median_us']
        res['gate']['batch_%d' % batch] = r
    info_sets = {'sparse_%d' % n: G.from_angles(shape, (np.arange(n) + 0.5 + 0.2 * np.sin(np.arange(n) + 1.0)) * (pi / n))
                 for n in (1, 2, 3, 4, 8)}
    info_sets['wedge_90deg_60'] = G.from_angle_range(shape, 60, 0.0, pi / 2)
    for batch in (8, 256):
        steps = {k: make_step(g, batch) for k, g in info_sets.items()}
        res['info']['batch_%d' % batch] = alternate(steps, max(3, a.reps // 2), a.iters)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
