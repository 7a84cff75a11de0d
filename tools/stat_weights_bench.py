"""Cost of measurement weights: the weighted data-consistency system against the unweighted one.

    python tools/stat_weights_bench.py [--reps 30] [--out FILE]

One operator (256 x 256, 60 views) and, for each case, the same call with and without per-sample weights W
(``v + gamma A*(W A v)``) timed alternately in one process: CUDA events around each call, and between calls the L2
is flushed (a 256 MB buffer, twice the B200's 126 MB of L2, is overwritten).  W is packed once before the timed
calls, as a sampler does.  Cases: ``normal_apply``, CG(5) (``cg_solve``) and ``dds_step`` (CG(5)) at B = 1, 8 and
256.  The JSON gives per case the median and spread (min, max) of the ``--reps`` calls of each variant and the
weighted / unweighted ratio of the medians, with the card's name and power limit.

Estimate (not a measurement): W adds (K + 1) * 4 * n_angles * n_det bytes per sample and DDS step (525 600 B at
K = 5), 2.4 % of the step's 22 022 720 algorithmic bytes at 256^2 / 60 views.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import diffusion_models_dev_project_b200 as pkg                                   # noqa: E402
from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D as G    # noqa: E402
from matched_adjoint_bench import FLUSH_BYTES, card                              # noqa: E402


def make_case(kind, rt, batch, weights, seed=0):
    geom = rt.geometry
    gen = torch.Generator(device='cuda').manual_seed(seed)
    img = lambda: torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen)      # noqa: E731
    x = img()
    if kind == 'normal_apply':
        return lambda: rt.normal_apply(x, 0.01, weights=weights)
    atb = rt.trafo_adjoint(rt(torch.rand(batch, 1, *geom.im_shape, device='cuda', generator=gen)))
    if kind == 'cg5':
        rhs = x + 0.01 * atb
        return lambda: rt.cg_solve(x, rhs, 0.01, 5, weights=weights)
    s, eps = img(), img()
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t = torch.full((batch,), 500., device='cuda')
    tp = torch.full((batch,), 490., device='cuda')
    return lambda: rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5, weights=weights)[0]


def alternate(calls, reps, flush):
    for fn in calls.values():                             # warm-up: module load, workspaces, packed weights
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps * len(calls))]
    i = 0
    for _ in range(reps):
        for k, fn in calls.items():
            flush.fill_(i & 0xff)
            a, b = ev[i]
            a.record()
            out = fn()
            b.record()
            times[k].append((a, b))
            i += 1
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    res = {}
    for k, v in times.items():
        us = np.array([a.elapsed_time(b) * 1e3 for a, b in v])
        res[k] = {'median_us': float(np.median(us)), 'min_us': float(us.min()), 'max_us': float(us.max()), 'calls': len(us)}
    res['weighted_over_unweighted'] = res['weighted']['median_us'] / res['unweighted']['median_us']
    return res


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--reps', type=int, default=30)
    p.add_argument('--out', default=None, help='also write the JSON here')
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('stat_weights_bench needs a CUDA device')
    flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device='cuda')
    geom = G.from_im_shape((256, 256), 60)
    rt = pkg.B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom)
    res = {'card': card(), 'timing': 'CUDA events per call, L2 flushed between calls, weighted / unweighted alternating',
           'cases': {}}
    for kind in ('normal_apply', 'cg5', 'dds_step'):
        for batch in (1, 8, 256):
            rng = np.random.default_rng(batch)
            w = torch.from_numpy(rng.uniform(0.1, 3.0, size=(batch, 1, *geom.obs_shape))).float().cuda()
            weights = pkg.MeasurementWeights(rt, w)
            name = '%s_256x256_60views_B%d' % (kind, batch)
            calls = {'unweighted': make_case(kind, rt, batch, None), 'weighted': make_case(kind, rt, batch, weights)}
            r = res['cases'][name] = alternate(calls, a.reps, flush)
            print('%-32s unweighted %9.1f us  weighted %9.1f us  ratio %.3f' % (
                name, r['unweighted']['median_us'], r['weighted']['median_us'], r['weighted_over_unweighted']),
                file=sys.stderr)
            del calls, weights
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
