"""Cost of the matched adjoint: pixel-driven against matched A*, and the operators built on it.

    python tools/matched_adjoint_bench.py [--reps 30] [--out FILE]

Two operators of the same geometry, ``B200RayTrafo(..., adjoint='pixel')`` and ``adjoint='matched'``, are timed
alternately in one process, one launch sequence at a time: CUDA events around each call, and between calls the L2
is flushed (a 256 MB buffer, twice the B200's 126 MB of L2, is overwritten) so that neither operator finds the
other's sinogram or image in the cache.  The JSON gives, per case, the median and the spread (min, max) of the
``--reps`` calls of each operator and the matched / pixel ratio of the medians:

  * A* (``trafo_adjoint``: sinogram re-layout + bp_tile) at 256 x 256, 60 views, B = 1, 8 and 256;
  * ``normal_apply`` (v + gamma A*A v), CG(5) (``cg_solve``) and ``dds_step`` (CG(5)) at B = 8 and 256;
  * A* of a 501 x 501 x 64-slice stack with 1200 views.

The card's name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import diffusion_models_dev_project_b200 as pkg                                   # noqa: E402
from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D as G    # noqa: E402

FLUSH_BYTES = 256 << 20


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = 'unknown'
    return {'name': name, 'power_limit_and_max_sm_clock': out}


def make_case(kind, geom, batch, adjoint, seed=0):
    rt = pkg.B200RayTrafo(geom.im_shape, geom.n_angles, geometry=geom, adjoint=adjoint)
    gen = torch.Generator(device='cuda').manual_seed(seed)
    img = lambda: torch.randn(batch, 1, *geom.im_shape, device='cuda', generator=gen)      # noqa: E731
    if kind == 'bp':
        y = torch.randn(batch, 1, *geom.obs_shape, device='cuda', generator=gen)
        return lambda: rt.trafo_adjoint(y)
    x = img()
    if kind == 'normal_apply':
        return lambda: rt.normal_apply(x, 0.01)
    atb = rt.trafo_adjoint(rt(torch.rand(batch, 1, *geom.im_shape, device='cuda', generator=gen)))
    if kind == 'cg5':
        rhs = x + 0.01 * atb
        return lambda: rt.cg_solve(x, rhs, 0.01, 5)
    s, eps = img(), img()
    abar = pkg.DDPM().alpha_bar_table('cuda')
    t = torch.full((batch,), 500., device='cuda')
    tp = torch.full((batch,), 490., device='cuda')
    return lambda: rt.dds_step(x, s, atb, eps, t, tp, abar, 0.01, 0.15, 5)[0]


def alternate(calls, reps, flush):
    for fn in calls.values():                             # warm-up: module load, workspaces
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
    res['matched_over_pixel'] = res['matched']['median_us'] / res['pixel']['median_us']
    return res


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--reps', type=int, default=30)
    p.add_argument('--out', default=None, help='also write the JSON here')
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('matched_adjoint_bench needs a CUDA device')
    flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device='cuda')
    g256 = G.from_im_shape((256, 256), 60)
    cases = [('bp', g256, b) for b in (1, 8, 256)]
    cases += [(k, g256, b) for k in ('normal_apply', 'cg5', 'dds_step') for b in (8, 256)]
    cases += [('bp', G.from_im_shape((501, 501), 1200), 64)]
    res = {'card': card(), 'timing': 'CUDA events per call, L2 flushed between calls, pixel / matched alternating',
           'cases': {}}
    for kind, geom, batch in cases:
        name = '%s_%dx%d_%dviews_B%d' % (kind, geom.n0, geom.n1, geom.n_angles, batch)
        calls = {adj: make_case(kind, geom, batch, adj) for adj in ('pixel', 'matched')}
        res['cases'][name] = alternate(calls, a.reps, flush)
        print('%-40s pixel %9.1f us  matched %9.1f us  ratio %.3f' % (
            name, res['cases'][name]['pixel']['median_us'], res['cases'][name]['matched']['median_us'],
            res['cases'][name]['matched_over_pixel']), file=sys.stderr)
        del calls
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
