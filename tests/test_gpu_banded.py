"""The peer-staged banded backprojection and band reduction of ``AngleShardedRayTrafo(reduce='peer')`` on one GPU.

``scd_bp_banded`` / ``scd_bp_il_banded`` store every backprojector tile of image band o as a dense
``[batch][band_rows][n1]`` slab into the staging buffer of the band's owner; ``scd_band_reduce`` adds the staged
copies in rank order and stores ``c_sum * sum + c_add * addend`` into up to 8 outputs.  Band and output addresses
are plain device addresses, so P local buffers stand in for P ranks' symmetric buffers: tests/banded_emulation.py
runs the ranks one after another through the Python wrappers (``_bp_banded``, ``_normal_banded``, ``_band_reduce``)
with the staging layout of ``sharding._PeerReduce.run`` (3 rotating staging buffers, slots sized for a chunk).

  * staged slabs bit-identical to ``_bp`` / ``normal_apply(add_identity=False)`` of the rank's angle range when
    both launches use whole tiles (``bp_rows=1``); ranks without angles store zeros;
  * every rank's result bit-identical to the float32 rank-order sum of those partials (plus ``v`` for A*A);
  * per-sample relative L2 error against the float64 oracle (weighted oracle on weighted view sets) at most 1e-5,
    also with the default tuning, where the result is also within 1e-6 of ``trafo_adjoint`` / ``normal_apply``;
  * 1 to 8 ranks, empty and short trailing bands, ragged sample groups, the packed path at batch 2, 8 / 16 / 32
    row tiles, more chunks than staging buffers, weighted views with ranks that own no angle;
  * angle ranges on weighted view sets through the NCCL path's operators (``_bp``, ``normal_apply``, ``_fp``);
  * ``band_reduce`` with general coefficients, 1 to 8 sources and 1 to 8 outputs against a numpy float32
    restatement (1 ulp);
  * no store outside a slab's rows, a chunk's samples or an owner's rows, checked with guarded NaN buffers;
  * invalid band layouts and reduction arguments rejected by the host-side checks, with a message, writing nothing.

Worst per-sample relative L2 error against float64, measured on an NVIDIA B200 at a 1000 W power limit (the same
with whole tiles and with the default tuning): A* of projected sinograms 1.6e-7 at 256^2, 9.2e-8 at 96x70 and 70x50,
1.4e-7 at 501^2, 6.2e-8 on the weighted view sets; ``v + gamma A*A v`` 1.7e-7, 9.2e-8, 1.7e-7 and 2.2e-7; at most
2.7e-7 from the unsharded operator.  NCCL path (white-noise sinograms): A* 1.3e-6, A*A 2.2e-7.  The file runs in
about 9 s there.

Not covered here, only by the two-GPU test (tests/test_gpu_multi.py): the multicast store (``multimem.st``, needs
NVSwitch), torch symmetric memory, and the cross-rank barriers of ``_PeerReduce.run``.
"""
import numpy as np
import pytest
import torch

import angle_set_oracle as W
import banded_emulation as E
import test_gpu_angle_sets as AS
import test_gpu_guards as TG
from conftest import rel_l2
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ORACLE_GATE = 1e-5          # per sample, as tests/test_gpu_multi.py
SAME_GATE = 1e-6            # default tuning against the unsharded operator
GAMMA = 0.05
NAN = float('nan')

UNIFORM = {'u256': ((256, 256), 60), 'u96x70': ((96, 70), 30), 'u70x50': ((70, 50), 9), 'u501': ((501, 501), 150)}


def _pkg():
    import diffusion_models_dev_project_b200 as pkg
    return pkg


def _sharding():
    from diffusion_models_dev_project_b200 import sharding
    return sharding


def _geometry(name):
    if name in UNIFORM:
        from diffusion_models_dev_project_b200.physics.geometry import ParallelBeamGeometry2D
        return ParallelBeamGeometry2D.from_im_shape(*UNIFORM[name])
    return AS._geometry(name)


def _ranges(name, rt, P):
    """Cost-balanced angle ranges as the sharded operator uses them; ``sparse3`` with equal counts, so that ranks
    3..P-1 own no angle."""
    sh = _sharding()
    if name == 'sparse3':
        return [sh.shard_range(rt.obs_shape[0], r, P) for r in range(P)]
    return sh.angle_cost_ranges(rt.angles, P)


def _partial(rt, op, data, rng):
    if op == 'bp':
        return rt._bp(data, rt.adj_scale, angle_range=rng)
    return rt.normal_apply(data, GAMMA, angle_range=rng, add_identity=False)


def _oracle(geom, op, data):
    og = W.geometry(geom)
    d = data.cpu().numpy()
    if op == 'bp':
        return W.bp(og, d)
    return d.astype(np.float64) + GAMMA * W.bp(og, O.fp(og, d))


def _per_sample(a, b):
    a = a.cpu().numpy() if torch.is_tensor(a) else a
    b = b.cpu().numpy() if torch.is_tensor(b) else b
    return np.array([rel_l2(a[i], b[i]) for i in range(a.shape[0])])


def _emulate(rt, L, n, ranges, op, data, staged=None):
    """The P ranks' results of one peer-reduced A* (op 'bp') or ``v + gamma A*A v`` (op 'normal') of ``data``."""
    dev, P = data.device, L.world
    stage = [torch.full((L.stage_floats,), NAN, device=dev) for _ in range(P)]
    result = [torch.full((n, 1, *rt.im_shape), NAN, device=dev) for _ in range(P)]

    def produce(r, lo, hi, ptrs, band_rows):
        if op == 'bp':
            rt._bp_banded(data[lo:hi], rt.adj_scale, ptrs, band_rows, angle_range=ranges[r])
        else:
            rt._normal_banded(data[lo:hi], GAMMA, ptrs, band_rows, angle_range=ranges[r])

    def reduce(stage_ptr, n_src, slot, batch, band_rows, rows, row_lo, outs, lo, hi):
        rt._band_reduce(stage_ptr, n_src, slot, batch, band_rows, rows, row_lo, outs, dev,
                        addend=data[lo:hi] if op == 'normal' else None, c_add=1.0 if op == 'normal' else 0.0)

    E.run(L, n, [s.data_ptr() for s in stage], [t.data_ptr() for t in result], produce, reduce,
          None if staged is None else (lambda c, lo, hi, buf: staged(stage, lo, hi, buf)))
    return result


# (geometry, ranks, slices, chunk, bp_tile)
CASES = [
    ('u256', 1, 1, 1, None),            # groups of one sample
    ('u256', 2, 2, 2, None),            # packed copy, V = 2
    ('u256', 3, 3, 3, None),            # one group of 4, one empty lane
    ('u256', 4, 8, 8, None),
    ('u256', 4, 8, 8, 8),
    ('u256', 4, 8, 8, 16),
    ('u256', 4, 8, 8, 32),
    ('u256', 8, 17, 17, None),          # two groups of 16, the second with 15 empty lanes
    ('u256', 2, 17, 4, None),           # 5 chunks (4, 4, 3, 3, 3): staging buffers reused, ragged groups
    ('u256', 3, 7, 2, None),            # 4 chunks (2, 2, 2, 1)
    ('u96x70', 4, 9, 2, None),          # width not a multiple of 32, last band empty
    ('u70x50', 8, 9, 2, None),          # five empty bands
    ('u501', 2, 3, 3, None),            # last band 245 of 256 rows
    ('u501', 8, 4, 2, None),            # last band 53 of 64 rows
    ('wedge90', 8, 8, 3, None),
    ('golden37', 4, 5, 2, None),        # view ids out of angular order
    ('sparse3', 8, 4, 1, None),         # ranks 3..7 own no angle
]


@pytest.mark.parametrize('op', ['bp', 'normal'])
@pytest.mark.parametrize('name,P,n,chunk,tile', CASES,
                         ids=['%s-P%d-n%d-c%d%s' % (c[:4] + ('-t%d' % c[4] if c[4] else '',)) for c in CASES])
def test_peer_staged_reduction_on_one_device(name, P, n, chunk, tile, op):
    geom = _geometry(name)
    rt = AS._rt(geom)
    dev = torch.device('cuda')
    L = E.Layout(geom.im_shape, P, chunk)
    ranges = _ranges(name, rt, P)
    gen = torch.Generator(device=dev).manual_seed(100 * P + n)
    data = torch.rand(n, 1, *geom.im_shape, device=dev, generator=gen)
    if op == 'bp':
        # a measured sinogram: white noise would make the comparison with the unsharded A* at other tile heights
        # (fp32 interpolation weights re-centred per tile) a 1.6e-6 affair, above SAME_GATE
        data = rt(data)
    ref = _oracle(geom, op, data)
    n1 = geom.im_shape[1]

    # whole tiles in both launches: the staged partials are the rank's own A* bit for bit
    rt.set_tuning(dev, bp_rows=1, bp_tile=tile or 0)
    want = torch.full((n, 1, *geom.im_shape), NAN, device=dev)

    def staged(stage, lo, hi, buf):
        parts = [_partial(rt, op, data[lo:hi], ranges[r]) for r in range(P)]
        for r, part in enumerate(parts):
            for o in range(P):
                row_lo, rows = L.band(o)
                slab = stage[o].view(E.NBUF, P, chunk, L.band_rows, n1)[buf, r, :hi - lo, :rows]
                assert torch.equal(slab, part[:, 0, row_lo:row_lo + rows]), ('slab', lo, r, o)
                if ranges[r][0] == ranges[r][1] and rows:
                    assert float(slab.abs().max()) == 0.0, ('empty range', r, o)
        acc = parts[0]
        for part in parts[1:]:
            acc = acc + part                         # rank order, float32
        want[lo:hi] = acc + data[lo:hi] if op == 'normal' else acc

    result = _emulate(rt, L, n, ranges, op, data, staged)
    assert not torch.isnan(want).any()
    for p in range(P):
        assert torch.equal(result[p], want), ('result', p)
    e_tiles = _per_sample(result[0], ref)

    # the default launch heuristics (tile heights balanced per launch)
    rt.set_tuning(dev, bp_rows=0, bp_tile=0)
    result = _emulate(rt, L, n, ranges, op, data)
    for p in range(1, P):
        assert torch.equal(result[p], result[0]), ('replica', p)
    e_default = _per_sample(result[0], ref)
    direct = rt.trafo_adjoint(data) if op == 'bp' else rt.normal_apply(data, GAMMA)
    e_direct = _per_sample(result[0], direct)
    print('\n%s %s P%d n%d: worst per-sample rel L2 vs fp64 %.2e (whole tiles) %.2e (default), vs unsharded %.2e'
          % (op, name, P, n, e_tiles.max(), e_default.max(), e_direct.max()))
    assert (e_tiles <= ORACLE_GATE).all(), e_tiles
    assert (e_default <= ORACLE_GATE).all(), e_default
    assert (e_direct <= SAME_GATE).all(), e_direct


# ------------------------------------------------------------------------------------------ NCCL path ---
@pytest.mark.parametrize('name,P', [('wedge90', 8), ('golden37', 4), ('golden37', 8), ('sparse3', 8)])
def test_weighted_angle_ranges_on_the_nccl_path(name, P):
    """``reduce='nccl'`` sums per-rank ``_bp`` / ``normal_apply`` results: their sums over the rank ranges must be
    the weighted operators, and every rank's rows of A must be those of the full A."""
    geom = _geometry(name)
    rt = AS._rt(geom)
    ranges = _ranges(name, rt, P)
    assert ranges[0][0] == 0 and ranges[-1][1] == geom.n_angles
    gen = torch.Generator(device='cuda').manual_seed(31)
    n = 5
    y = torch.randn(n, 1, *geom.obs_shape, device='cuda', generator=gen)
    x = torch.rand(n, 1, *geom.im_shape, device='cuda', generator=gen)
    z = rt._bp(y, rt.adj_scale, angle_range=ranges[0])
    nrm = rt.normal_apply(x, GAMMA, angle_range=ranges[0], add_identity=True)
    for r in range(1, P):
        z = z + rt._bp(y, rt.adj_scale, angle_range=ranges[r])
        nrm = nrm + rt.normal_apply(x, GAMMA, angle_range=ranges[r], add_identity=False)
    e_bp, e_n = _per_sample(z, _oracle(geom, 'bp', y)), _per_sample(nrm, _oracle(geom, 'normal', x))
    print('\nnccl %s P%d: worst per-sample rel L2 vs fp64: A* %.2e, normal %.2e' % (name, P, e_bp.max(), e_n.max()))
    assert (e_bp <= ORACLE_GATE).all(), e_bp
    assert (e_n <= ORACLE_GATE).all(), e_n
    full = rt(x)
    for lo, hi in ranges:
        yl = rt._fp(x, angle_range=(lo, hi))
        assert torch.equal(yl[:, :, lo:hi], full[:, :, lo:hi])
        assert float(yl[:, :, :lo].abs().sum()) == 0.0 and float(yl[:, :, hi:].abs().sum()) == 0.0


# --------------------------------------------------------------------------------------- band_reduce ---
@pytest.mark.parametrize('n_src,n_out', [(1, 1), (3, 3), (8, 8), (5, 2)])
def test_band_reduce_with_general_coefficients(n_src, n_out):
    """``out_p[rows] = c_sum * (stage_0 + ... + stage_{n-1}) + c_add * addend[rows]`` for every output p, against
    numpy in float32 (rank-order sum, rounded product); 1 ulp for the fused multiply-add, which numpy rounds
    twice.  Slab rows past ``rows`` and samples past ``batch`` are NaN: reading them would show."""
    rt = _pkg().B200RayTrafo((70, 50), 9)
    dev = torch.device('cuda')
    n0, n1, band_rows, batch, chunk = 70, 50, 32, 3, 4
    gen = torch.Generator(device=dev).manual_seed(n_src * 10 + n_out)
    stage = torch.full((n_src, chunk, band_rows, n1), NAN, device=dev)
    addend = 10.0 * torch.randn(batch, 1, n0, n1, device=dev, generator=gen)
    c_sum, c_add = np.float32(0.37), np.float32(-1.9)
    for row_lo, rows in ((64, 6), (32, 32), (0, 17)):
        stage.fill_(NAN)
        stage[:, :batch, :rows] = torch.randn(n_src, batch, rows, n1, device=dev, generator=gen)
        acc = np.zeros((batch, rows, n1), dtype=np.float32)
        for r in range(n_src):
            acc = acc + stage[r, :batch, :rows].cpu().numpy()
        scaled = c_sum * acc                                                     # float32 product
        a = addend[:, 0, row_lo:row_lo + rows].cpu().numpy()
        fused = (np.float64(c_add) * a.astype(np.float64) + scaled.astype(np.float64)).astype(np.float32)
        for with_addend in (False, True):
            outs = [torch.full((batch, n0, n1), NAN, device=dev) for _ in range(n_out)]
            rt._band_reduce(stage.data_ptr(), n_src, chunk * band_rows * n1, batch, band_rows, rows, row_lo,
                            [o.data_ptr() for o in outs], dev, addend=addend if with_addend else None,
                            c_add=float(c_add), c_sum=float(c_sum))
            for o in outs:
                got = o[:, row_lo:row_lo + rows].cpu().numpy()
                if with_addend:
                    assert (np.abs(got - fused) <= np.spacing(np.abs(fused))).all(), (row_lo, rows)
                else:
                    np.testing.assert_array_equal(got, scaled)
                assert torch.isnan(o[:, :row_lo]).all() and torch.isnan(o[:, row_lo + rows:]).all()


# ------------------------------------------------------------------------------- writes outside buffers ---
# (geometry, ranks, batch, slot size in slices): every ragged group fits in the slot
GUARD_CASES = [('u96x70', 4, 3, 4), ('u256', 3, 5, 8), ('u256', 8, 17, 32), ('u70x50', 8, 9, 16), ('u501', 8, 2, 3)]


@pytest.mark.parametrize('op', ['bp', 'normal'])
@pytest.mark.parametrize('name,P,batch,chunk', GUARD_CASES, ids=['%s-P%d-b%d-c%d' % c for c in GUARD_CASES])
def test_banded_stores_stay_inside_their_rows(name, P, batch, chunk, op):
    """Staging slots (one buffer per owner, slots for ``chunk`` > ``batch`` slices) and results (one sample more
    than the batch) start as NaN between guard regions.  A rank's call writes rows ``[0, rows)`` of samples
    ``< batch`` of its slot in every owner's buffer and nothing else; an owner's reduction writes its rows of
    samples ``< batch`` of every result and nothing else."""
    geom = _geometry(name)
    rt = AS._rt(geom)
    dev = torch.device('cuda')
    n0, n1 = geom.im_shape
    L = E.Layout(geom.im_shape, P, chunk)
    ranges = _ranges(name, rt, P)
    gen = torch.Generator(device=dev).manual_seed(batch)
    if op == 'bp':
        data = torch.randn(batch, 1, *geom.obs_shape, device=dev, generator=gen)
    else:
        data = torch.rand(batch, 1, *geom.im_shape, device=dev, generator=gen)
    stage = [TG.Guarded(P * L.slot * 4, dev) for _ in range(P)]
    results = [TG.Guarded((batch + 1) * n0 * n1 * 4, dev) for _ in range(P)]
    for r in range(P):
        ptrs = [s.ptr + r * L.slot * 4 for s in stage]
        if op == 'bp':
            rt._bp_banded(data, rt.adj_scale, ptrs, L.band_rows, angle_range=ranges[r])
        else:
            rt._normal_banded(data, GAMMA, ptrs, L.band_rows, angle_range=ranges[r])
        torch.cuda.synchronize()
        for o, s in enumerate(stage):
            rows = L.band(o)[1]
            st = s.floats(P, chunk, L.band_rows, n1)
            assert torch.isfinite(st[r, :batch, :rows]).all(), ('unwritten', r, o)
            assert torch.isnan(st[r, :batch, rows:]).all(), ('rows past the band', r, o)
            assert torch.isnan(st[r, batch:]).all(), ('samples past the batch', r, o)
            assert torch.isnan(st[r + 1:]).all(), ('next slot', r, o)
            assert s.intact(), ('guard', r, o)
    done = torch.zeros(n0, dtype=torch.bool, device=dev)
    for o in range(P):
        row_lo, rows = L.band(o)
        if rows == 0:
            continue
        rt._band_reduce(stage[o].ptr, P, L.slot, batch, L.band_rows, rows, row_lo, [g.ptr for g in results], dev,
                        addend=data if op == 'normal' else None, c_add=1.0 if op == 'normal' else 0.0)
        torch.cuda.synchronize()
        done[row_lo:row_lo + rows] = True
        for p, g in enumerate(results):
            f = g.floats(batch + 1, n0, n1)
            assert torch.isfinite(f[:batch, done]).all(), ('unwritten', o, p)
            assert torch.isnan(f[:batch, ~done]).all(), ('other owners\' rows', o, p)
            assert torch.isnan(f[batch:]).all(), ('samples past the batch', o, p)
            assert g.intact(), ('guard', o, p)
    assert bool(done.all())


# ---------------------------------------------------------------------------------------- error paths ---
def test_invalid_band_arguments_are_rejected_and_write_nothing():
    """Arguments the host-side checks reject: ``SCD_E_INVALID``, a message naming the problem, no store into any
    band, output or the caller's scratch (``scd_bp_banded`` checks the band layout before it re-lays out the
    sinogram).  An empty batch or an empty band is no work: 0, nothing written."""
    import ctypes as C
    from diffusion_models_dev_project_b200 import _lib
    lib = _lib.load()
    rt = _pkg().B200RayTrafo((256, 256), 60)
    dev = torch.device('cuda')
    h = rt._handle(dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    n0, n1, na = 256, 256, 60
    P, batch = 2, 3
    L = E.Layout((n0, n1), P, batch)
    gen = torch.Generator(device=dev).manual_seed(5)
    y = torch.randn(batch, 1, *rt.obs_shape, device=dev, generator=gen)
    x = torch.rand(batch, 1, n0, n1, device=dev, generator=gen)
    scr = TG.Guarded(lib.scd_bp_scratch_bytes(h.ptr, batch), dev)
    qp, _ = rt._aligned(rt._fp_il(x))
    stage = [TG.Guarded(P * L.slot * 4, dev) for _ in range(P)]
    outs = [TG.Guarded(batch * n0 * n1 * 4, dev) for _ in range(P)]
    good = [s.ptr for s in stage]
    torch.cuda.synchronize()

    def bp(ptrs, n_bands, band_rows, b=batch):
        return lib.scd_bp_banded(h.ptr, y.data_ptr(), b, 0, na, rt.adj_scale, rt._ptr_array(ptrs), n_bands, band_rows,
                                 scr.ptr, scr.nbytes, st)

    def bp_il(ptrs, n_bands, band_rows, b=batch, sino_il=qp):
        return lib.scd_bp_il_banded(h.ptr, sino_il, b, 0, na, rt.adj_scale, rt._ptr_array(ptrs), n_bands, band_rows,
                                    st)

    def reduce(ptrs, n_out=None, b=batch, band_rows=128, rows=128, row_lo=0, multicast=0):
        return lib.scd_band_reduce(good[0], P, L.slot, b, band_rows, rows, n1, row_lo, n0, rt._ptr_array(ptrs),
                                   len(ptrs) if n_out is None else n_out, multicast, None, 0.0, 1.0, st)

    def rejected(rc, what):
        assert rc == _lib.SCD_E_INVALID, (rc, what)
        assert what in _lib.last_error(), (_lib.last_error(), what)

    for call in (bp, bp_il):
        rejected(call(good, P, 0), 'bad band layout')
        rejected(call(good, P, 48), 'bad band layout')
        rejected(call(good, P, 64), 'bad band layout')                  # 2 x 64 rows < 256
        rejected(call(good, 0, 128), '1..8 bands')
        rejected(call(good * 5, 9, 128), '1..8 bands')
        rejected(call([good[0], 0], P, 128), 'null band pointer')
        assert call(good, P, 128, b=0) == 0
    rejected(bp_il(good, P, 128, sino_il=qp + 4), '128-byte aligned')
    res = [o.ptr for o in outs]
    rejected(reduce(res, rows=129), 'bad argument')                     # rows > band_rows
    rejected(reduce(res, row_lo=200), 'bad argument')                   # row_lo + rows > n0
    rejected(reduce(res, n_out=0), 'bad argument')
    rejected(reduce(res * 5, n_out=9), 'bad argument')
    rejected(reduce(res, multicast=1), 'multicast')
    rejected(reduce([res[0], 0]), 'null output pointer')
    assert reduce(res, b=0) == 0 and reduce(res, rows=0) == 0
    torch.cuda.synchronize()
    for g in stage + outs + [scr]:
        assert g.intact() and torch.isnan(g.floats(g.nbytes // 4)).all()
