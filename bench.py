#!/usr/bin/env python
"""Benchmark of the DDS / SCD data-consistency hot path on B200 (contract: see the task brief).

Workload (BASELINE.json configs[1]): "AAPM 256x256 sparse-view (60 angles) DDS-style sampling
with CG data consistency, batch 8 on 1 B200": 256x256 images, 60 angles x 365 detector bins,
DDPM schedule, 100 reverse steps per sample, CG with 5 iterations, gamma 0.01, eta 0.15, the
full-size guided-diffusion UNet as the (PyTorch) score caller, synthetic disk-ellipse phantoms,
random-init weights.

One bench *step* = one reverse-diffusion step of the whole batch: score call, then the hot path
(Tweedie -> rhs -> CG(5): 6 A + 6 A* + vector updates -> DDIM: 19 launches).  A sample needs 100 of them, so
    value [samples/s] = n_gpus * batch / (100 * seconds_per_step).
Multi-GPU: one process per GPU, the sample batch is sharded, no data-path collective (weak scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the predictor returned in the last timed step (x_next, xhat0) as float32 .npy files;
the inputs depend only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import functools
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IM, ANGLES, NDET = 256, 60, 365
REVERSE_STEPS = 100
CG_ITER, GAMMA, ETA = 5, 0.01, 0.15
# algorithmic bytes per sample (fp32), SURVEY.md section 8(d) / BASELINE.md section 4
BYTES = {
    'fp_march': 4 * (IM * IM + ANGLES * NDET),
    'bp_tile': 4 * (IM * IM + ANGLES * NDET),
    'bp_tile_axpy_dot': 4 * (2 * IM * IM + ANGLES * NDET),      # + read of the addend
    'cg_update_xr': 6 * 4 * IM * IM,
    'cg_direction_update': 3 * 4 * IM * IM,        # p = r + beta p (fused into the backprojector's epilogue)
    'tweedie_rhs': 5 * 4 * IM * IM,
    'ddim': 4 * 4 * IM * IM,
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=8, help='samples per GPU')
    ap.add_argument('--unet', default='aapm', choices=['aapm', 'small'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--kernel-batch', type=int, default=256, help='batch of the large-batch kernel sweep')
    ap.add_argument('--no-extra', action='store_true',
                    help='skip the config 3 / 4 / 5 blocks (stack_501, hot_path_sweep, adapted)')
    ap.add_argument('--cpu-threads', type=int, default=0,
                    help='host threads of the CPU reference arm (0 = every core this process may use)')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='write the outputs of the last timed step (x_next, xhat0) to DIR/<name>.npy, for either '
                         '--impl (float32, at most 64 MB in all)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    return args


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(out_dir, arrays, rank=0, world=1):
    """Save the [batch, ...] tensors of `arrays` as float32 DIR/<name>.npy (suffix _rank<r> when sharded).  When they
    would exceed DUMP_BYTES over all ranks, the same seeded subset of samples is kept in every array."""
    os.makedirs(out_dir, exist_ok=True)
    n = next(iter(arrays.values())).shape[0]
    per_sample = sum(4 * t[0].numel() for t in arrays.values())
    keep = min(n, DUMP_BYTES // world // per_sample)
    assert keep > 0, 'one sample of the outputs (%d bytes) exceeds the dump limit of %d bytes per rank' \
        % (per_sample, DUMP_BYTES // world)
    idx = None if keep == n else torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, keep, replace=False)))
    suffix = '_rank%d' % rank if world > 1 else ''
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        np.save(os.path.join(out_dir, name + suffix + '.npy'), (t if idx is None else t[idx]).numpy())


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)['hbm_gbs']), 'measured'
    return 6650.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


def measured_traffic():
    """DRAM bytes per launch of our kernels at the bench batch, from the latest ncu capture
    committed under profiles/ (rNN_traffic.json); None when no capture is available."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r*_traffic.json')))
    if not files:
        return None, None
    with open(files[-1]) as f:
        return json.load(f), os.path.basename(files[-1])


def time_pairs():
    from diffusion_models_dev_project_b200 import _schedule_jump
    ts = _schedule_jump(REVERSE_STEPS, 1, 1)
    skip = 1000 // REVERSE_STEPS
    return [(i * skip, j * skip if j > 0 else -1) for i, j in zip(ts[:-1], ts[1:])]


def make_unet(kind):
    from bench_support.adm_unet import aapm_unet, small_unet
    torch.manual_seed(0)
    return (aapm_unet() if kind == 'aapm' else small_unet()).eval()


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def build_id():
    """sha256 (16 hex digits) of the native library the bench loaded and of the sources it was built from, so that a
    stale .so cannot be benchmarked unnoticed."""
    import hashlib
    from diffusion_models_dev_project_b200 import _lib, build as b
    h = hashlib.sha256()
    with open(_lib.LIB_PATH, 'rb') as f:
        h.update(f.read())
    hs = hashlib.sha256()
    for src in [os.path.join(b.CSRC, n) for n in b.SOURCES] + list(b.HEADERS):
        with open(src, 'rb') as f:
            hs.update(f.read())
    return {'lib_sha16': h.hexdigest()[:16], 'src_sha16': hs.hexdigest()[:16], 'stale': bool(b.needs_build())}


# ------------------------------------------------------------------ CPU arm ---
def cpu_reference_arm(args, steps, warmup, quiet=False):
    """The reference's CPU path for one reverse step at batch 1 (its MatmulRayTrafo handles one
    image per call, reference src/physics/matmul_ray_trafo.py:108-109): torch.sparse.mm projector
    + the reference's cg / Tweedie / ddim recurrences + the same UNet on the host cores.
    Uses the reference's own code when SCD_REFERENCE_ROOT names a checkout of it, else the oracle port.  Returns the
    timings and, under 'outputs', what the last timed step returned (x_next, xhat0)."""
    from oracle import oracle as O
    from oracle import ref_harness
    from bench_support.phantoms import disk_ellipses
    torch.set_grad_enabled(False)
    # torch.distributed.run exports OMP_NUM_THREADS=1: pin the thread count explicitly so that the CPU arm
    # means the same thing at every N (only rank 0 runs it, so it may use every core of the box)
    cores = args.cpu_threads if args.cpu_threads > 0 else host_cores()
    torch.set_num_threads(cores)
    cores = torch.get_num_threads()
    geom = O.OracleGeometry((IM, IM), ANGLES)
    ort = O.OracleRayTrafo(geom)
    score = make_unet(args.unet)
    x0 = torch.from_numpy(disk_ellipses(1, IM, seed=1))
    y = ort(x0)
    atb = ort.trafo_adjoint(y)
    pairs = time_pairs()
    torch.manual_seed(1)
    x = torch.randn(1, 1, IM, IM)
    kind = 'port'
    if ref_harness.available():
        src = ref_harness.import_reference()           # noqa: F841
        from src.samplers.utils import decomposed_diffusion_sampling_sde_predictor as ref_dds
        from src.utils.sde import DDPM as RefDDPM
        sde = RefDDPM()
        kind = 'reference'

        def one(x, t, tp):
            return ref_dds(score=score, sde=sde, x=x, rhs=atb, time_step=(torch.ones(1) * t, torch.ones(1) * tp),
                           eta=ETA, gamma=GAMMA, step_size=1, cg_kwargs={'max_iter': CG_ITER}, ray_trafo=ort)
    else:
        abar = O.ref_port_alpha_bar()

        def one(x, t, tp):
            return O.ref_port_dds_step(score, x, atb, abar, torch.ones(1) * t, torch.ones(1) * tp, GAMMA, ETA,
                                       CG_ITER, ort)
    for i in range(warmup):
        x, xm = one(x, *pairs[i % len(pairs)])
    t0 = time.perf_counter()
    for i in range(steps):
        x, xm = one(x, *pairs[(warmup + i) % len(pairs)])
    dt = (time.perf_counter() - t0) / max(steps, 1)
    # projector alone, for the per-operator comparison
    ta = time.perf_counter(); ort(x); ta = time.perf_counter() - ta
    tb = time.perf_counter(); ort.trafo_adjoint(y); tb = time.perf_counter() - tb
    # data-consistency part alone (no score model): Tweedie + CG(5) + DDIM on the host
    zero_score = lambda x, t: torch.zeros_like(x)                                      # noqa: E731
    abar_p = O.ref_port_alpha_bar()
    dc = time.perf_counter()
    O.ref_port_dds_step(zero_score, x, atb, abar_p, torch.ones(1) * 500., torch.ones(1) * 490., GAMMA, ETA, CG_ITER, ort)
    dc = time.perf_counter() - dc
    return {'value': 1.0 / (REVERSE_STEPS * dt), 'unit': 'samples/s', 'cores': cores, 'kind': kind,
            'sample': '%d reverse step(s) at batch 1 (of %d per sample): %s UNet + 6 A + 6 A* (torch.sparse.mm) + '
                      'CG/DDIM on host; %.2f s/step; A %.3f s, A* %.3f s per apply'
                      % (steps, REVERSE_STEPS, args.unet, dt, ta, tb),
            'seconds_per_step': dt, 'fp_seconds': ta, 'bp_seconds': tb,
            'dc_seconds': dc, 'outputs': {'x_next': x, 'xhat0': xm}}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    cb = cpu_reference_arm(args, steps, warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cb['outputs'])
    line = {
        'impl': 'reference', 'metric': 'SCD samples/sec at 256^2', 'value': cb['value'], 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': steps, 'warmup': warm, 'ms_per_step': cb['seconds_per_step'] * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, batch=1),
        'cpu_baseline': {k: cb[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
        'e2e': {'value': cb['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'host': {'cores_used': cb['cores'], 'cores_available': host_cores(),
                 'omp_num_threads_env': os.environ.get('OMP_NUM_THREADS')},
        'data_consistency_only': {'seconds_per_step_batch1': cb['dc_seconds'],
                                  'samples_per_s': 1.0 / (REVERSE_STEPS * cb['dc_seconds']),
                                  'note': 'Tweedie + CG(5) (6 A + 6 A*) + DDIM on the host, no score model: the part '
                                          'this repository replaces'},
    }
    print(json.dumps(line))


def workload_config(args, batch):
    return {'workload': 'AAPM-shape 256x256, 60 angles x 365 bins, DDS sampling, CG(%d), gamma %g, eta %g, '
                        '%d reverse steps per sample, %s UNet score caller (random init)'
                        % (CG_ITER, GAMMA, ETA, REVERSE_STEPS, args.unet),
            'batch_per_gpu': batch, 'reverse_steps_per_sample': REVERSE_STEPS, 'cg_iter': CG_ITER,
            'step': 'one reverse-diffusion step of the whole batch (score + Tweedie + CG + DDIM)',
            'l2': 'working set per step (UNet activations, >1 GB at batch 8) exceeds the 126 MB L2; '
                  'kernel sweep flushes L2 between launches',
            'parallelism': 'sample-sharded, no collective'}


# ------------------------------------------------------------------ GPU arm ---
def cuda_time(fn, iters, flush=None):
    """Average device time of fn() in ms, CUDA events on the current stream, optional L2 flush
    (a write larger than L2) before every launch, outside the timed interval."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in evs:
        if flush is not None:
            flush.zero_()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in evs]))


def kernel_sweep(rt, batch, dev, hbm_peak, iters=20):
    """Per-kernel device time and algorithmic GB/s at one batch size (L2 flushed before each launch)."""
    from diffusion_models_dev_project_b200 import fused, DDPM
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(batch, 1, IM, IM, device=dev, generator=gen)
    p = torch.rand(batch, 1, IM, IM, device=dev, generator=gen)
    s = torch.randn(batch, 1, IM, IM, device=dev, generator=gen)
    y = rt(x)
    abar = DDPM().alpha_bar_table(dev)
    t = torch.ones(batch, device=dev) * 500.
    tp = torch.ones(batch, device=dev) * 490.
    out = {}
    q_il = rt._fp_il(x)                                                    # interleaved sinogram of x (as inside CG)
    lead = x.shape[:-2]
    x_il = rt._img_il(x)                                                   # sample-interleaved image (as inside CG)
    p_il = rt._img_il(p)
    d_il = torch.empty_like(p_il)
    cases = {
        'il_pack+fp_march': lambda: rt._fp_il(x),                          # 2 launches: interleaving pass + march
        'fp_march': lambda: rt._fp_ilimg(x_il, batch),                     # 1 launch: A of an interleaved image
        'bp_tile': lambda: rt._bp_il(q_il, lead, rt.adj_scale),            # 1 launch
        'bp_tile_il_axpy': lambda: rt._bp_ilimg(q_il, batch, 0.01 * rt.adj_scale, addend_il=p_il, addend_scale=1.0,
                                                out_il=d_il),              # 1 launch, interleaved in and out
        'bp_tile_axpy_dot': lambda: rt._bp_il(q_il, lead, 0.01 * rt.adj_scale, addend=p, addend_scale=1.0),
        'A_public': lambda: rt._fp(x),                                     # public trafo: pack + march (user layout out)
        'Aadj_public': lambda: rt._bp(y, rt.adj_scale),                    # public trafo_adjoint: sino_pack + bp_tile
        'tweedie_rhs': lambda: fused.tweedie_rhs(x, s, t, abar, atb=p, gamma=GAMMA),
        'ddim': lambda: fused.ddim_ddpm(x, s, p, t, tp, abar, ETA),
    }
    BYTES.update({'il_pack+fp_march': BYTES['fp_march'], 'A_public': BYTES['fp_march'], 'Aadj_public': BYTES['bp_tile'],
                  'bp_tile_il_axpy': BYTES['bp_tile_axpy_dot']})
    for name, fn in cases.items():
        for _ in range(3):
            fn()
        ms = cuda_time(fn, iters, flush)
        gbs = BYTES[name] * batch / (ms * 1e-3) / 1e9
        out[name] = {'ms': ms, 'GB/s': gbs, 'frac_hbm': gbs / hbm_peak}
    # whole CG solve (6 A + 6 A* + 5 update_xr; direction updates ride on the backprojector's epilogue)
    op = rt.normal_op(GAMMA)
    from diffusion_models_dev_project_b200 import cg
    for _ in range(3):
        cg(op, x, p, CG_ITER)
    ms = cuda_time(lambda: cg(op, x, p, CG_ITER), iters, flush)
    cg_bytes = (CG_ITER + 1) * (BYTES['fp_march'] + BYTES['bp_tile_axpy_dot']) + CG_ITER * BYTES['cg_update_xr'] \
        + (CG_ITER - 1) * BYTES['cg_direction_update']
    gbs = cg_bytes * batch / (ms * 1e-3) / 1e9
    out['cg_solve_k5'] = {'ms': ms, 'GB/s': gbs, 'frac_hbm': gbs / hbm_peak}
    del flush
    return out


def run_b200(args):
    import torch.distributed as dist
    import diffusion_models_dev_project_b200 as pkg
    from diffusion_models_dev_project_b200 import fused
    from bench_support.phantoms import disk_ellipses

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl b200 needs a CUDA device (there is no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    torch.set_grad_enabled(False)
    hbm_peak, peak_kind = peaks()
    B = args.batch

    # ---- setup (untimed): operator, schedule, score caller, synthetic measurements ----
    rt = pkg.B200RayTrafo((IM, IM), ANGLES)
    sde = pkg.DDPM()
    score = make_unet(args.unet).to(dev)
    gt = torch.from_numpy(disk_ellipses(B, IM, seed=1 + rank)).to(dev)
    y = pkg.simulate(gt, rt, 0.01, rng=np.random.default_rng(1 + rank))
    atb = rt.trafo_adjoint(y)
    pairs = time_pairs()
    ones = torch.ones(B, device=dev)
    torch.manual_seed(1 + rank)
    x = sde.prior_sampling([B, 1, IM, IM]).to(dev)
    predictor = functools.partial(pkg.decomposed_diffusion_sampling_sde_predictor, score=score, sde=sde, rhs=atb,
                                  cg_kwargs={'max_iter': CG_ITER}, eta=ETA, gamma=GAMMA, use_simplified_eqn=True,
                                  ray_trafo=rt, step_size=1)

    def step(x, i):
        t, tp = pairs[i % len(pairs)]
        return predictor(x=x, time_step=(ones * t, ones * tp))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: W warm-up + exactly K steps ----
    for i in range(args.warmup):
        x, xm = step(x, i)
    barrier()
    fused.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        for i in range(args.steps):
            x, xm = step(x, args.warmup + i)
        e1.record()
        barrier()
    launches = fused.launch_count()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'x_next': x, 'xhat0': xm}, rank, world)
    ms_total = e0.elapsed_time(e1)
    tt = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_step = float(tt.item()) / args.steps
    value = world * B / (REVERSE_STEPS * ms_step * 1e-3)

    # ---- end-to-end through the public predictor API with HOST buffers ----
    hx = torch.empty(B, 1, IM, IM).pin_memory()
    hx.copy_(x.cpu())
    hatb = atb.cpu().pin_memory()
    hout = torch.empty(2, B, 1, IM, IM).pin_memory()
    dx, datb = torch.empty_like(x), torch.empty_like(atb)

    def e2e_step(i):
        dx.copy_(hx, non_blocking=True)
        datb.copy_(hatb, non_blocking=True)
        t, tp = pairs[i % len(pairs)]
        xn, xh = pkg.decomposed_diffusion_sampling_sde_predictor(
            score=score, sde=sde, x=dx, rhs=datb, time_step=(ones * t, ones * tp), eta=ETA, gamma=GAMMA,
            step_size=1, cg_kwargs={'max_iter': CG_ITER}, use_simplified_eqn=True, ray_trafo=rt)
        hout[0].copy_(xn, non_blocking=True)
        hout[1].copy_(xh, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        hx.copy_(hout[0])
    for i in range(min(args.warmup, 3)):
        e2e_step(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        e2e_step(args.warmup + i)
    e1.record()
    barrier()
    te = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    ms_e2e = float(te.item()) / args.steps
    e2e = {'value': world * B / (REVERSE_STEPS * ms_e2e * 1e-3), 'unit': 'samples/s',
           'h2d_bytes_per_step': int(2 * B * IM * IM * 4), 'd2h_bytes_per_step': int(2 * B * IM * IM * 4),
           'ms_per_step': ms_e2e}

    # ---- hot path alone (no score call): the part this repo implements ----
    s_fix = torch.randn(B, 1, IM, IM, device=dev)
    eps_fix = torch.randn(B, 1, IM, IM, device=dev)
    abar = sde.alpha_bar_table(dev)

    def dc_only():
        rt.dds_step(x, s_fix, atb, eps_fix, ones * 500., ones * 490., abar, GAMMA, ETA, CG_ITER)
    for _ in range(5):
        dc_only()
    fused.launch_count(reset=True)
    dc_only()
    dc_launches = fused.launch_count()
    ms_dc = cuda_time(dc_only, 20)
    dc_bytes = (CG_ITER + 1) * (BYTES['fp_march'] + BYTES['bp_tile_axpy_dot']) + CG_ITER * BYTES['cg_update_xr'] \
        + (CG_ITER - 1) * BYTES['cg_direction_update'] + BYTES['tweedie_rhs'] + BYTES['ddim']

    # ---- the other BASELINE configurations (all ranks take part: config 4 has a collective) ----
    extra = {}
    if not args.no_extra:
        from bench_support import config_blocks as CB
        score = None
        torch.cuda.empty_cache()
        extra['hot_path_sweep'] = CB.sweep_block(dev, world, rank)
        extra['stack_501'] = CB.stack_block(dev, world, rank)
        extra['adapted'] = CB.adapted_block(dev, world, rank)
        score = None

    line = None
    if rank == 0:
        sweep_small = kernel_sweep(rt, B, dev, hbm_peak)
        sweep_big = kernel_sweep(rt, args.kernel_batch, dev, hbm_peak) if args.kernel_batch else {}
        dom = max(('fp_march', 'bp_tile_axpy_dot'), key=lambda k: sweep_small[k]['ms'])
        traffic, traffic_src = measured_traffic()
        tr, pipe = None, None
        if traffic is not None and B == 8:
            names = ['fp_march_kernel'] if dom == 'fp_march' else ['bp_tile_kernel']
            if all(n in traffic for n in names):
                tr = sum(traffic[n]['dram_bytes_per_launch'] for n in names)
                pipe = traffic[names[-1]].get('shared_pipe_frac')
        roofline = {'bound': 'hbm', 'kernel': dom + ' (one launch)',
                    'achieved': sweep_small[dom]['GB/s'], 'peak': hbm_peak,
                    'unit': 'GB/s', 'frac': sweep_small[dom]['frac_hbm'], 'traffic': tr,
                    'traffic_source': traffic_src,
                    'peak_source': peak_kind + ' (MEASURED_PEAKS.json hbm_gbs, burst copy)' if peak_kind == 'measured'
                    else 'fallback 6.65 TB/s',
                    'algorithmic_bytes_per_launch': BYTES[dom] * B, 'launch_ms': sweep_small[dom]['ms'],
                    'shared_memory_pipe_frac_ncu': pipe,
                    'note': 'A/A* are bound by the shared-memory pipe (8 B per tap pair and sample), not HBM: '
                            'DESIGN.md section 4; large-batch figures in kernels_b%d.  The kernel is timed on a '
                            'sample-interleaved image, the form it has inside CG (scd_fp_ilimg: one launch, no packed copy); '
                            'traffic is its DRAM traffic under ncu (cold caches): the image once, the sinogram once'
                            % args.kernel_batch}
        line = {
            'metric': 'SCD samples/sec at 256^2', 'value': value, 'unit': 'samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, B), 'e2e': e2e, 'gpu_launches': int(launches),
            'gpu_launches_per_step': launches / max(args.steps, 1),
            'roofline': roofline,
            'hot_path': {'ms_per_step': ms_dc, 'launches_per_step': int(dc_launches),
                         'share_of_step': ms_dc / ms_step, 'samples_per_s_hot_path_only':
                             B / (REVERSE_STEPS * ms_dc * 1e-3),
                         'GB/s': dc_bytes * B / (ms_dc * 1e-3) / 1e9,
                         'frac_hbm': dc_bytes * B / (ms_dc * 1e-3) / 1e9 / hbm_peak},
            'kernels_b%d' % B: sweep_small, 'kernels_b%d' % args.kernel_batch: sweep_big,
            'clocks': clk.summary(),
            'build': build_id(),
        }
        line.update(extra)
    if world > 1:
        dist.barrier()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            score = None
            torch.cuda.empty_cache()
            cb = cpu_reference_arm(args, steps=2, warmup=1)
            line['cpu_baseline'] = {k: cb[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
            line['hot_path']['vs_cpu_data_consistency_only'] = cb['dc_seconds'] / (ms_dc * 1e-3 / B)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_b200(a)
