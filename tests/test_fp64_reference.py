"""CPU tests of the float64 reference of the DDS step (tests/fp64_reference.py): it agrees with the reference's
own outputs (golden vectors) and with the float32 port of the reference's code, and it is sharp enough to tell
apart the mistakes a kernel could make (an alpha-bar index one off, another sample's time step, one CG iteration
too few) -- each of those lands far outside the 2e-5 gate the GPU tests apply."""
import numpy as np
import pytest

from conftest import rel_l2
from fp64_reference import (BENCH_PAIR, abar_at, cg64, ddim64, dds_step64, matrices, port_dds_step, time_steps,
                            tweedie64)
from oracle import oracle as O

GATE = 2e-5          # x_next of the GPU tests against dds_step64 at gamma = 0.01


def _abar():
    return O.ref_port_alpha_bar().numpy()


def test_abar_index_truncates_and_clamps():
    ab = _abar()
    assert ab.shape == (1001,) and ab[0] == 1.0
    got = abar_at(ab, np.array([250.6, 0., -1., 999., 2000., -7.], dtype=np.float32))
    assert np.array_equal(got, ab[[251, 1, 0, 1000, 1000, 0]].astype(np.float64))


@pytest.mark.parametrize('gamma', [0.01, 1.0])
def test_cg64_matches_reference_cg(golden, gamma):
    """cg64 against the reference's own cg on the oracle operator (tests/golden/make_golden.py:cg_fixture):
    fp32 round-off apart at gamma = 0.01; at gamma = 1 the fp32 recurrences amplify round-off, still < 1e-3."""
    d = golden('cg_small.npz')
    geom = O.OracleGeometry(tuple(int(v) for v in d['im']), int(d['num_angles']))
    for k in (0, 1, 2, 5):
        got = cg64(geom, d['x0'], d['rhs'], gamma, k)
        assert got.dtype == np.float64 and got.shape == d['x0'].shape
        ref = d['x_g%g_k%d' % (gamma, k)]
        for b in range(ref.shape[0]):
            assert rel_l2(got[b], ref[b]) < (1e-5 if gamma < 0.1 else 1e-3), (gamma, k, b, rel_l2(got[b], ref[b]))


def test_tweedie64_and_ddim64_match_reference(golden):
    """Against apTweedy / ddim of the reference's own code (tests/golden/tweedie_ddim.npz: every sample shares the
    time step, so the batch-wide and the per-sample NaN rules agree; case (300, 310) has a NaN tbeta)."""
    d = golden('tweedie_ddim.npz')
    ab = _abar()
    for ci, (t, tp) in enumerate(d['cases']):
        tt, tpp = np.full(3, t, np.float32), np.full(3, tp, np.float32)
        assert rel_l2(tweedie64(d['x'], d['s'], tt, ab), d['tweedie_%d' % ci]) < 1e-6, ci
        for eta in (0.0, 0.15, 0.85):
            got = ddim64(d['xhat'], d['s'], d['noise_%d' % ci], tt, tpp, ab, eta)
            assert rel_l2(got, d['ddim_%d_%g' % (ci, eta)]) < 1e-6, (ci, eta)


@pytest.fixture(scope='module')
def step():
    """256 x 256, 60 angles, batch 8: disk-ellipse phantoms, seeded N(0, 1) x / s / eps, the eight time pairs."""
    from bench_support.phantoms import disk_ellipses
    geom = O.OracleGeometry((256, 256), 60)
    J, Bm = matrices(geom)
    gt = disk_ellipses(8, 256, seed=3)
    atb = (Bm @ (J @ gt.reshape(8, -1).T.astype(np.float64))).T.reshape(gt.shape).astype(np.float32)
    rng = np.random.default_rng(4)
    x, s, eps = (rng.standard_normal(gt.shape).astype(np.float32) for _ in range(3))
    t, tp = time_steps(8)
    args = dict(x=x, s=s, atb=atb, eps=eps, t=t, t_prev=tp, abar=_abar(), gamma=0.01, eta=0.15, n_iter=5)
    return geom, args, port_dds_step(geom, **args)


def test_dds_step64_matches_port(step):
    """dds_step64 against O.ref_port_dds_step (fp32, the reference's code) per sample, one sample at a time."""
    geom, args, (port_next, port_xh0) = step
    x_next, xhat0 = dds_step64(geom, **args)
    assert np.isfinite(x_next).all()
    for b in range(8):
        assert rel_l2(xhat0[b], port_xh0[b]) < 1e-6, b
        assert rel_l2(x_next[b], port_next[b]) < 1e-5, (b, rel_l2(x_next[b], port_next[b]))


def _shifted_table(ab):
    """abar[trunc(t) + 2]: the alpha-bar index one step late."""
    return np.append(ab[1:], ab[-1])


@pytest.mark.parametrize('variant', ['abar_index_plus_1', 'sample0_times', 'one_cg_iteration_less'])
def test_wrong_steps_fail_the_gate(step, variant):
    """Each mistake moves every sample it changes by more than 5x the GPU gate away from the port."""
    geom, args, (port_next, _) = step
    args = dict(args)
    changed = list(range(8))
    if variant == 'abar_index_plus_1':
        args['abar'] = _shifted_table(args['abar'])
    elif variant == 'sample0_times':
        args['t'] = np.full(8, args['t'][0], np.float32)
        args['t_prev'] = np.full(8, args['t_prev'][0], np.float32)
        changed = list(range(1, 8))                   # the eight pairs differ
    else:
        args['n_iter'] -= 1
    x_next, _ = dds_step64(geom, **args)
    errs = [rel_l2(x_next[b], port_next[b]) for b in changed]
    assert min(errs) > 5 * GATE, (variant, errs)


def test_uniform_time_step_rules_agree(step):
    """At the bench's pair (every sample at (500, 490)) the batched port and dds_step64 agree as well: there the
    reference's batch-wide NaN rule and the per-sample one coincide."""
    geom, args, _ = step
    args = dict(args)
    args['t'], args['t_prev'] = time_steps(8, pairs=(BENCH_PAIR,))
    import torch
    from fp64_reference import port_trafo
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))          # noqa: E731
    s = T(args['s'])
    port_next, _ = O.ref_port_dds_step(lambda *_: s, T(args['x']), T(args['atb']), T(args['abar']), T(args['t']),
                                       T(args['t_prev']), args['gamma'], args['eta'], args['n_iter'], port_trafo(geom),
                                       noise=T(args['eps']))
    x_next, _ = dds_step64(geom, **args)
    for b in range(8):
        assert rel_l2(x_next[b], port_next[b].numpy()) < 1e-5, b
