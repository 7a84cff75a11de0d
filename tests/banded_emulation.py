"""One-device emulation of the peer-staged band reduction (helper module of the tests, not a test file).

``AngleShardedRayTrafo(reduce='peer')`` sums the angle-sharded backprojections of P GPUs on the backprojector
itself: rank r stores the tiles of image band o straight into slot ``[buf][r]`` of owner o's staging buffer
(``scd_bp_banded`` / ``scd_bp_il_banded``), then owner o adds the P staged copies of its band in rank order and
stores the sum into every rank's result (``scd_band_reduce``).  Band and result addresses are plain device
addresses, so on one GPU P local buffers can stand in for the P ranks' symmetric buffers: :func:`run` calls the
same kernels, one rank after another, with the staging layout of ``sharding._PeerReduce.run`` -- slots sized for
``chunk`` slices, ``NBUF`` rotating staging buffers, results written at slice offset ``lo`` of every chunk.

The two callables are injected so that the layout arithmetic can be checked on the CPU with numpy stand-ins
(tests/test_banded_layout_cpu.py) and the kernels on the GPU (tests/test_gpu_banded.py).
"""
from types import SimpleNamespace

from diffusion_models_dev_project_b200.sharding import AngleShardedRayTrafo, _PeerReduce, band_layout

NBUF = _PeerReduce.NBUF
F32 = 4                                   # bytes per element of the staging and result buffers


class Layout:
    """Band and staging geometry of P ranks for an ``n0 x n1`` image and slice chunks of at most ``chunk``."""

    def __init__(self, im_shape, world, chunk):
        self.n0, self.n1 = int(im_shape[0]), int(im_shape[1])
        self.world, self.chunk = int(world), int(chunk)
        self.band_rows = band_layout(self.n0, self.world)
        self.slot = self.chunk * self.band_rows * self.n1            # floats per (buffer, source rank)
        self.stage_floats = NBUF * self.world * self.slot             # one owner's staging buffer

    def band(self, owner):
        """``(row_lo, rows)`` of the band ``owner`` reduces (``rows`` may be 0: empty trailing band)."""
        row_lo = min(self.n0, owner * self.band_rows)
        return row_lo, max(0, min(self.n0, (owner + 1) * self.band_rows) - row_lo)

    def chunks(self, n):
        """The slice chunks ``[(lo, hi)]`` the sharded operator uses for a stack of ``n`` slices."""
        return AngleShardedRayTrafo._chunk_bounds(SimpleNamespace(chunk=self.chunk), n)

    def slot_offset(self, buf, src):
        """Element offset of slot ``[buf][src]`` in an owner's staging buffer (dense ``[chunk][band_rows][n1]``)."""
        return (buf * self.world + src) * self.slot


def run(layout, n, stage_ptrs, result_ptrs, bp_banded, band_reduce, staged=None):
    """Emulate one call of ``_PeerReduce.run`` over ``n`` slices on one device.

    ``stage_ptrs[o]`` / ``result_ptrs[p]``: base addresses of owner o's staging buffer (``layout.stage_floats``
    floats) and of rank p's result (``n * n0 * n1`` floats).
    ``bp_banded(rank, lo, hi, band_ptrs, band_rows)``: rank's banded backprojection of slices ``[lo, hi)``.
    ``band_reduce(stage_ptr, n_src, slot_stride, batch, band_rows, rows, row_lo, out_ptrs, lo, hi)``: one owner's
    reduction of chunk ``[lo, hi)`` (the caller adds the addend rows ``[lo, hi)`` for the normal operator).
    ``staged(c, lo, hi, buf)``: called once every rank has stored chunk c, before the owners reduce it."""
    P, L = layout.world, layout
    for c, (lo, hi) in enumerate(L.chunks(n)):
        buf = c % NBUF
        for r in range(P):
            bp_banded(r, lo, hi, [stage_ptrs[o] + L.slot_offset(buf, r) * F32 for o in range(P)], L.band_rows)
        if staged is not None:
            staged(c, lo, hi, buf)
        for o in range(P):
            row_lo, rows = L.band(o)
            if rows > 0:
                outs = [result_ptrs[p] + lo * L.n0 * L.n1 * F32 for p in range(P)]
                band_reduce(stage_ptrs[o] + L.slot_offset(buf, 0) * F32, P, L.slot, hi - lo, L.band_rows, rows, row_lo,
                            outs, lo, hi)
