"""The fused DDS data-consistency step (`B200RayTrafo.dds_step`, scd_dds_step) and the fused CG (`cg` on a
`NormalOp`, scd_cg) against the float64 reference of tests/fp64_reference.py, on every path the step takes:

  * the interleaved-image path (batch >= 3, and batch 1 when the image width is a multiple of 4): tweedie_il ->
    cg_run_il (fp_march with the beta recurrence in its output phase, bp_tile's mode-1 epilogue,
    cg_update_xr_il) -> ddim_il, in groups of 4, 8 or 16 samples, with empty lanes and several groups;
  * groups of one sample: the plain-layout Tweedie / CG update / DDIM kernels of vec_ops.cu;
  * the packed-copy path (batch 2, batch 1 with n1 % 4 != 0, or `fp_source=1`): Tweedie fused into the pack pass
    of the first projection (fp_packq mode 2), the direction update into the later ones (mode 1).

Every sample has its own (t, t_prev) (fp64_reference.TIME_PAIRS), so a kernel that reads another sample's time
step, or another group's partial sums, fails here.  Run with -s to see the worst per-sample error of each run."""
import collections

import numpy as np
import pytest
import torch

from conftest import rel_l2
from fp64_reference import BENCH_PAIR, TIME_PAIRS, cg64, dds_step64, port_dds_step, time_steps
from oracle import oracle as O

pytestmark = pytest.mark.gpu

BENCH = (0.01, 0.15, 5)                                      # (gamma, eta, n_iter) of bench.py
MORE = ((0.01, 0.0, 0), (0.01, 1.0, 1), (1.0, 0.15, 5))      # for the untuned 256 x 256 cases
XHAT0_GATE = 1e-6
X_NEXT_GATE = 2e-5                                           # at gamma = 0.01

Case = collections.namedtuple('Case', 'shape angles batch tune il group')
CASES = [
    # shape, angles, batch, tuning, il path, samples per group
    Case((256, 256), 60, 8, {}, True, 8),                    # the bench: one group of 8
    Case((256, 256), 60, 1, {}, True, 1),                    # one sample per group: plain-layout kernels
    Case((256, 256), 60, 2, {}, False, 2),                   # packed path
    Case((256, 256), 60, 3, {}, True, 4),                    # one empty lane
    Case((256, 256), 60, 17, {}, True, 16),                  # two groups, the last with one sample
    Case((256, 256), 60, 40, {}, True, 16),                  # three groups
    Case((96, 70), 13, 1, {}, False, 1),                     # packed at batch 1 (n1 % 4 != 0)
    Case((96, 70), 13, 6, {}, True, 8),                      # ragged 128-pixel row tile
    Case((501, 501), 24, 5, {}, True, 8),                    # largest strips, odd sizes
    Case((256, 256), 60, 8, {'fp_source': 1}, False, 8),     # packed path at the bench batch
    Case((256, 256), 60, 8, {'fp_samples': 1}, True, 1),     # 8 groups of one: plain-layout kernels over a batch
    Case((256, 256), 60, 8, {'fp_samples': 4}, True, 4),     # two groups of 4
    Case((256, 256), 60, 3, {'fp_samples': 16}, True, 16),   # 13 empty lanes
]


def _case_id(c):
    return '%dx%d-a%d-b%d' % (*c.shape, c.angles, c.batch) + ''.join('-%s=%d' % kv for kv in c.tune.items())


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


_PHANTOMS = {}


def _phantoms(shape, n=4):
    """``n`` disk-ellipse phantoms of ``shape`` (centre crop of square ones)."""
    g = _PHANTOMS.get(shape)
    if g is None:
        from bench_support.phantoms import disk_ellipses
        m = max(shape)
        sq = disk_ellipses(n, m, seed=5)
        o0, o1 = (m - shape[0]) // 2, (m - shape[1]) // 2
        g = _PHANTOMS[shape] = np.ascontiguousarray(sq[..., o0:o0 + shape[0], o1:o1 + shape[1]])
    return g


def _inputs(rt, batch, seed=0):
    """Seeded N(0, 1) ``x``, ``s``, ``eps`` and ``atb = A*(A gt)`` of phantoms (cycled over the batch)."""
    gen = torch.Generator(device='cuda').manual_seed(seed)
    x, s, eps = (torch.randn(batch, 1, *rt.im_shape, device='cuda', generator=gen) for _ in range(3))
    ph = _phantoms(rt.im_shape)
    gt = torch.from_numpy(ph[[b % len(ph) for b in range(batch)]]).cuda()
    return x, s, rt.trafo_adjoint(rt(gt)), eps


def _errs(a, b):
    """Per-sample relative L2 distance of ``a`` from ``b``."""
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    return np.array([rel_l2(a[i], b[i]) for i in range(len(b))])


def _watched(batch, group):
    """The first and the last sample and the two samples either side of every group boundary."""
    out = {0, batch - 1}
    for k in range(group, batch, group):
        out |= {k - 1, k}
    return sorted(out)


@pytest.mark.parametrize('case', CASES, ids=[_case_id(c) for c in CASES])
def test_dds_step_matches_fp64(case):
    """Per run: the path is the one the case names; xhat0 is bit-identical to scd_tweedie_rhs; for n_iter = 0
    x_next is bit-identical to scd_ddim; xhat0 and x_next match dds_step64 per sample; the inputs are unchanged.
    Gates: xhat0 1e-6; x_next 2e-5 at gamma = 0.01.  At gamma = 1 the system is ill-conditioned and fp32 round-off
    is amplified by the recurrences (the fp32 port reaches 1e-4 of fp64 on some samples), so there the gate is
    the rule of test_cg_matches_reference_cg: no further from fp64 than 4x the port's own distance + 1e-5.  The
    floor is 1e-5, not less: the port's distance is one draw of round-off and lands anywhere from 1e-7 to 3e-4
    per sample, while the kernels sit at 3e-6 .. 1.6e-5 on every sample (B200); with a floor of 1e-6 a sample on
    which the port happens to land close to fp64 gets a gate below fp32 noise (batch 40, sample 0: 5.10e-6 against
    a gate of 5.09e-6).  The gamma = 0.01 runs of every case keep the fixed 2e-5 gate.
    Then batch independence: watched samples run alone (default tuning: the batch-1 path) agree with their
    in-batch result to 1e-5 at gamma = 0.01; at gamma = 1 to twice the fp64 gate (both results lie within it)."""
    pkg = _pkg()
    from diffusion_models_dev_project_b200 import fused
    dev = torch.device('cuda')
    rt = pkg.B200RayTrafo(case.shape, case.angles)
    geom = O.OracleGeometry(case.shape, case.angles)
    abar = pkg.DDPM().alpha_bar_table(dev)
    ab = abar.cpu().numpy()
    B = case.batch
    x, s, atb, eps = _inputs(rt, B)
    host = dict(x=x.cpu().numpy(), s=s.cpu().numpy(), atb=atb.cpu().numpy(), eps=eps.cpu().numpy())
    untuned_256 = case.shape == (256, 256) and not case.tune
    runs = [(p, TIME_PAIRS) for p in (BENCH,) + (MORE if untuned_256 else ())] + [(BENCH, (BENCH_PAIR,))]
    done = []
    rt.set_tuning('cuda', **case.tune)
    try:
        assert rt.il_supported(B, 'cuda') == case.il
        for (gamma, eta, n_iter), pairs in runs:
            t_np, tp_np = time_steps(B, pairs)
            t, tp = torch.from_numpy(t_np).to(dev), torch.from_numpy(tp_np).to(dev)
            args = (x, s, atb, eps, t, tp, abar)
            before = [a.clone() for a in args]
            x_next, xhat0 = rt.dds_step(x, s, atb, eps, t, tp, abar, gamma, eta, n_iter)
            assert all(torch.equal(a, b) for a, b in zip(args, before)), 'dds_step changed an input'
            assert torch.equal(xhat0, fused.tweedie_rhs(x, s, t, abar))
            if n_iter == 0:
                assert torch.equal(x_next, fused.ddim_ddpm(xhat0, s, eps, t, tp, abar, eta))
            ref_next, ref_xh0 = dds_step64(geom, t=t_np, t_prev=tp_np, abar=ab, gamma=gamma, eta=eta, n_iter=n_iter,
                                           **host)
            e_xh, e_next = _errs(xhat0, ref_xh0), _errs(x_next, ref_next)
            if gamma <= 0.01:
                gate = np.full(B, X_NEXT_GATE)
            else:
                port_next, _ = port_dds_step(geom, t=t_np, t_prev=tp_np, abar=ab, gamma=gamma, eta=eta,
                                             n_iter=n_iter, **host)
                gate = 4 * _errs(port_next, ref_next) + 1e-5
            print('\ndds_step %s gamma=%g eta=%g n_iter=%d t=%s: worst per-sample rel L2 vs fp64: xhat0 %.2e, '
                  'x_next %.2e (sample %d, gate %.1e)' % (_case_id(case), gamma, eta, n_iter,
                                                          'per-sample' if len(pairs) > 1 else 'bench',
                                                          e_xh.max(), e_next.max(), int(e_next.argmax()),
                                                          gate[e_next.argmax()]))
            assert (e_xh <= XHAT0_GATE).all(), e_xh
            assert (e_next <= gate).all(), (e_next, gate)
            done.append((gamma, eta, n_iter, t, tp, x_next, gate))
    finally:
        rt.set_tuning('cuda', **{k: 0 for k in case.tune})
    for gamma, eta, n_iter, t, tp, x_next, gate in done:
        for b in _watched(B, case.group):
            one = [a[b:b + 1].clone() for a in (x, s, atb, eps, t, tp)]
            solo, _ = rt.dds_step(*one, abar, gamma, eta, n_iter)
            err = rel_l2(solo.cpu().numpy(), x_next[b:b + 1].cpu().numpy())
            limit = 1e-5 if gamma <= 0.01 else 2 * gate[b]
            assert err <= limit, (b, gamma, eta, n_iter, err, limit)


@pytest.mark.parametrize('batch', [17, 40])
def test_cg_several_groups_matches_fp64(batch):
    """scd_cg with two and three groups of 16 against cg64, per sample.  Sample b is scaled by 10^((b % 5) - 2),
    so the per-sample partial sums (||r||^2, <p,d>) differ by up to eight orders of magnitude between samples:
    a partial sum read from the wrong sample or group gives a far wrong alpha or beta."""
    pkg = _pkg()
    rt = pkg.B200RayTrafo((256, 256), 60)
    geom = O.OracleGeometry((256, 256), 60)
    assert rt.il_supported(batch, 'cuda')
    x, _, atb, _ = _inputs(rt, batch, seed=1)
    scale = torch.tensor([10.0 ** ((b % 5) - 2) for b in range(batch)], device='cuda').view(-1, 1, 1, 1)
    x0 = x * scale
    rhs = (x + 0.01 * atb) * scale
    x0_np, rhs_np = x0.cpu().numpy(), rhs.cpu().numpy()
    for k in (1, 2, 5):
        out = pkg.cg(rt.normal_op(0.01), x0, rhs, k)
        e = _errs(out, cg64(geom, x0_np, rhs_np, 0.01, k))
        print('\ncg batch %d k=%d: worst per-sample rel L2 vs fp64 %.2e (sample %d)' % (batch, k, e.max(), int(e.argmax())))
        assert (e <= X_NEXT_GATE).all(), (k, e)
    assert np.array_equal(x0.cpu().numpy(), x0_np) and np.array_equal(rhs.cpu().numpy(), rhs_np)


def test_zero_sample_stays_in_its_lane():
    """Batch 8 (one group of 8): sample 5 has x = s = atb = 0, so its residual is exactly zero and CG divides 0/0
    -- NaN, as the reference's cg gives (no guard, like the kernels).  The NaN must stay in its lane of the
    interleaved images, sinograms and partial sums: the other seven samples are finite and match fp64."""
    pkg = _pkg()
    dev = torch.device('cuda')
    rt = pkg.B200RayTrafo((256, 256), 60)
    geom = O.OracleGeometry((256, 256), 60)
    abar = pkg.DDPM().alpha_bar_table(dev)
    ab = abar.cpu().numpy()
    x, s, atb, eps = _inputs(rt, 8, seed=2)
    for v in (x, s, atb):
        v[5] = 0
    t_np, tp_np = time_steps(8)
    gamma, eta, n_iter = BENCH
    x_next, xhat0 = rt.dds_step(x, s, atb, eps, torch.from_numpy(t_np).to(dev), torch.from_numpy(tp_np).to(dev),
                                abar, gamma, eta, n_iter)
    host = dict(x=x.cpu().numpy(), s=s.cpu().numpy(), atb=atb.cpu().numpy(), eps=eps.cpu().numpy())
    only5 = {k: v[5:6] for k, v in host.items()}
    port5, _ = port_dds_step(geom, t=t_np[5:6], t_prev=tp_np[5:6], abar=ab, gamma=gamma, eta=eta, n_iter=n_iter,
                             **only5)
    assert np.isnan(port5).all()
    assert bool(torch.isnan(x_next[5]).all())
    assert bool((xhat0[5] == 0).all())
    ref_next, ref_xh0 = dds_step64(geom, t=t_np, t_prev=tp_np, abar=ab, gamma=gamma, eta=eta, n_iter=n_iter, **host)
    others = [b for b in range(8) if b != 5]
    assert bool(torch.isfinite(x_next[others]).all())
    e_xh = _errs(xhat0[others], ref_xh0[others])
    e_next = _errs(x_next[others], ref_next[others])
    print('\nzero sample 5: worst rel L2 of the other samples vs fp64: xhat0 %.2e, x_next %.2e' % (e_xh.max(), e_next.max()))
    assert (e_xh <= XHAT0_GATE).all() and (e_next <= X_NEXT_GATE).all(), (e_xh, e_next)
