"""The offset arithmetic of the one-device peer-reduction emulation (tests/banded_emulation.py), on the CPU.

The driver is test logic that the GPU tests of the banded backprojector rely on: if it put a rank's slab at the
wrong slot, a chunk's result at the wrong slice or an owner's rows at the wrong offset, those tests would check the
kernels against a wrong layout.  Here it runs with numpy stand-ins for the two kernels: the stand-in backprojector
copies the oracle's partial image rows into flat staging arrays by element offset, the stand-in reduction adds the
staged copies in rank order.  The assembled stack must equal the float32 rank-order sum of the oracle partials bit
for bit (and the full oracle backprojection to float32 rounding), for every world size, image shape and chunk count
the GPU tests use; staging rows no rank writes must stay NaN."""
import numpy as np
import pytest

import banded_emulation as E
from conftest import rel_l2
from oracle import oracle as O
from diffusion_models_dev_project_b200.sharding import angle_cost_ranges, shard_range


class FlatMemory:
    """Flat float32 arrays (NaN-filled) at made-up device addresses; an address resolves to an array slice."""

    def __init__(self):
        self.arrays = []

    def alloc(self, n):
        base = (len(self.arrays) + 1) << 40
        self.arrays.append((base, np.full(int(n), np.nan, dtype=np.float32)))
        return base

    def view(self, addr, count):
        for base, arr in self.arrays:
            if base <= addr < base + arr.size * 4:
                off, rem = divmod(addr - base, 4)
                assert rem == 0 and off + count <= arr.size, 'access past the end of a buffer'
                return arr[off:off + count]
        raise AssertionError('address %#x is in no buffer' % addr)


# (image shape, angles, world size, slices, chunk, ranges): every configuration of tests/test_gpu_banded.py
CASES = [
    ((256, 256), 60, 1, 1, 1, 'cost'),
    ((256, 256), 60, 2, 2, 2, 'cost'),
    ((256, 256), 60, 3, 3, 3, 'cost'),
    ((256, 256), 60, 4, 8, 8, 'cost'),
    ((256, 256), 60, 8, 17, 17, 'cost'),
    ((256, 256), 60, 2, 17, 4, 'cost'),          # 5 chunks of 4, 4, 3, 3, 3: staging buffers reused
    ((256, 256), 60, 3, 7, 2, 'cost'),           # 4 chunks of 2, 2, 2, 1
    ((256, 256), 60, 8, 8, 3, 'cost'),           # 3 chunks of 3, 3, 2
    ((256, 256), 37, 4, 5, 2, 'cost'),
    ((96, 70), 30, 4, 9, 2, 'cost'),             # last band empty
    ((70, 50), 9, 8, 9, 2, 'cost'),              # five empty bands
    ((501, 501), 150, 2, 3, 3, 'cost'),          # last band 245 of 256 rows
    ((501, 501), 150, 8, 4, 2, 'cost'),          # last band 53 of 64 rows
    ((256, 256), 3, 8, 4, 1, 'count'),           # five ranks without angles
]


@pytest.mark.parametrize('shape,na,P,n,chunk,ranges', CASES,
                         ids=['%dx%d-a%d-P%d-n%d-c%d' % (c[0] + c[1:5]) for c in CASES])
def test_emulated_peer_reduction_assembles_the_oracle_backprojection(shape, na, P, n, chunk, ranges):
    og = O.OracleGeometry(shape, na)
    n0, n1 = shape
    L = E.Layout(shape, P, chunk)
    rng = np.random.default_rng(P * 1000 + n)
    y = rng.standard_normal((n, *og.obs_shape)).astype(np.float32)
    parts = angle_cost_ranges(og.angles, P) if ranges == 'cost' else [shard_range(na, r, P) for r in range(P)]
    partial = [O.bp(og, y, angle_range=parts[r]) for r in range(P)]
    mem = FlatMemory()
    stage = [mem.alloc(L.stage_floats) for _ in range(P)]
    result = [mem.alloc(n * n0 * n1) for _ in range(P)]
    calls = {'bp': 0, 'reduce': 0}

    def bp_banded(r, lo, hi, ptrs, band_rows):
        assert len(ptrs) == P and band_rows == L.band_rows and hi - lo <= chunk
        for i, p in enumerate(ptrs):
            k0, k1 = min(n0, i * band_rows), min(n0, (i + 1) * band_rows)
            slab = mem.view(p, (hi - lo) * band_rows * n1).reshape(hi - lo, band_rows, n1)
            slab[:, :k1 - k0] = partial[r][lo:hi, k0:k1]
        calls['bp'] += 1

    def band_reduce(stage_ptr, n_src, slot_stride, batch, band_rows, rows, row_lo, out_ptrs, lo, hi):
        assert 0 < rows <= band_rows and row_lo + rows <= n0 and len(out_ptrs) == P
        acc = np.zeros((batch, rows, n1), dtype=np.float32)
        for r in range(n_src):
            slab = mem.view(stage_ptr + r * slot_stride * 4, batch * band_rows * n1).reshape(batch, band_rows, n1)
            acc = acc + slab[:, :rows]
        for p in out_ptrs:
            mem.view(p, batch * n0 * n1).reshape(batch, n0, n1)[:, row_lo:row_lo + rows] = acc
        calls['reduce'] += 1

    E.run(L, n, stage, result, bp_banded, band_reduce)
    n_chunks = len(L.chunks(n))
    assert n_chunks == -(-n // chunk)
    owners = sum(L.band(o)[1] > 0 for o in range(P))
    assert calls == {'bp': P * n_chunks, 'reduce': owners * n_chunks}
    want = partial[0].copy()
    for r in range(1, P):
        want = want + partial[r]
    full = O.bp(og, y)
    for p in range(P):
        got = mem.view(result[p], n * n0 * n1).reshape(n, n0, n1)
        np.testing.assert_array_equal(got, want)
        assert max(rel_l2(got[b], full[b]) for b in range(n)) < 1e-6
    # every rank fills its slot of each buffer up to the largest chunk that used it (the first: chunks are
    # levelled, larger ones first); slab rows past the image and samples past that chunk are never written
    sizes = [hi - lo for lo, hi in L.chunks(n)]
    for o in range(P):
        rows = L.band(o)[1]
        st = mem.view(stage[o], L.stage_floats).reshape(E.NBUF, P, chunk, L.band_rows, n1)
        assert np.isnan(st[:, :, :, rows:]).all()
        for b in range(E.NBUF):
            m = sizes[b] if b < n_chunks else 0
            assert not np.isnan(st[b, :, :m, :rows]).any()
            assert np.isnan(st[b, :, m:]).all()


def test_layout_matches_the_peer_reduction_of_the_sharded_operator():
    """Band rows, owner rows and chunks are those of sharding._PeerReduce / AngleShardedRayTrafo."""
    L = E.Layout((501, 501), 8, 128)
    assert L.band_rows == 64 and [L.band(o) for o in (0, 6, 7)] == [(0, 64), (384, 64), (448, 53)]
    assert [hi - lo for lo, hi in L.chunks(501)] == [126, 125, 125, 125]
    assert L.slot == 128 * 64 * 501 and L.stage_floats == 3 * 8 * L.slot
    L2 = E.Layout((70, 50), 8, 2)
    assert [L2.band(o) for o in range(8)] == [(0, 32), (32, 32), (64, 6)] + [(70, 0)] * 5
    assert E.Layout((96, 70), 4, 1).band(3) == (96, 0)
