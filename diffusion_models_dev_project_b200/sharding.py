"""Multi-GPU partitioning of the hot path (one process per GPU, torch.distributed).

Two cases (SURVEY.md section 8e; the reference itself is single-process, single-GPU):

* **Sample / slice batches** -- every sample's A, A*, CG and DDIM is independent (the CG
  reductions are per sample, reference src/utils/cg.py:22,27,33), so the batch is split into
  contiguous shards and no collective touches the data path: :func:`shard_range`.

* **One large slice stack, angle-sharded** -- rank r owns the contiguous angles ``[lo_r, hi_r)``, chosen so that
  every rank carries the same projector + backprojector cost (:func:`angle_cost_ranges`).
  ``A``: each rank computes only its sinogram rows (no communication; the other rows of the
  returned tensor are zero).  ``A*``: each rank backprojects its rows into a full-size partial
  image stack and the partials are summed with an all-reduce (NCCL over NVLink on the GPU box).
  The stack is processed in slice chunks so that the all-reduce of chunk c overlaps the
  backprojection of chunk c+1.  CG vectors are replicated, so every dot product is local.

  With ``reduce='peer'`` (CUDA, one box) the sum rides on the backprojector instead: the image rows are
  split into one band per rank, the backprojector's epilogue stores every tile straight into the memory
  of the band's owner (torch symmetric memory: peer buffers mapped into every rank, stores travel over
  NVLink / NVSwitch while the kernel computes its other tiles), the owner adds the staged copies in rank
  order and stores the result into every rank's output (``scd_bp_banded`` / ``scd_band_reduce``).  The two
  cross-GPU ordering points per chunk are stream-ordered NCCL barriers on a side stream.

The wrapped operator only has to provide ``_fp(x, angle_range=)``, ``_bp(y, scale,
angle_range=)``, ``adj_scale``, ``im_shape`` and ``obs_shape`` -- :class:`B200RayTrafo` does;
the CPU tests drive the same code with an oracle-backed stand-in over ``gloo``.
"""
import os

import torch
import torch.distributed as dist
from torch import Tensor


def shard_range(n: int, rank: int, world: int):
    """Contiguous ``[lo, hi)`` share of ``n`` items for ``rank``; sizes differ by at most one."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def angle_cost_ranges(angles, world: int, fp_weight: float = 1.75):
    """Contiguous angle ranges ``[(lo, hi)] * world`` of (nearly) equal COST instead of equal count.

    The ray-driven projector skips the part of every ray that misses the image, so an angle costs it in proportion
    to ``max(|cos phi|, |sin phi|)`` (the number of (row, ray) pairs inside the square): angles near the axes are
    ~40 % dearer than angles near the diagonals.  The pixel-driven backprojector costs the same for every angle.
    ``cost_i = fp_weight * max(|cos|, |sin|) / 0.9 + 1`` with ``fp_weight`` = time of A over time of A* per angle
    (measured ~1.75 on the 501^2 stack).  With equal counts over 8 ranks the two outer and the two middle ranks carry
    the dear angles and set the time of A for everyone."""
    import numpy as np
    a = np.asarray(angles, dtype=np.float64)
    n = len(a)
    if world <= 1 or n < world:
        return [shard_range(n, r, world) for r in range(world)]
    cost = fp_weight * np.maximum(np.abs(np.cos(a)), np.abs(np.sin(a))) / 0.9 + 1.0
    cum = np.concatenate([[0.0], np.cumsum(cost)])
    bounds = [0]
    for r in range(1, world):
        target = cum[-1] * r / world
        k = int(np.searchsorted(cum, target))
        k = k if abs(cum[k] - target) <= abs(cum[k - 1] - target) else k - 1
        bounds.append(min(max(k, bounds[-1] + 1), n - (world - r)))          # every rank keeps at least one angle
    bounds.append(n)
    return [(bounds[r], bounds[r + 1]) for r in range(world)]


class AngleShardedRayTrafo:
    """Angle-sharded view of a ray transform.

    ``trafo``            -> this rank's rows of ``A x`` (others zero) -- stays sharded.
    ``trafo_adjoint``    -> ``A* y`` summed over ranks (y: full-shape sinogram whose rows outside
                            this rank's range are ignored).
    ``normal_apply``     -> ``v + gamma * A*(A v)`` with one all-reduce per call.  With ``reduce='peer'`` the
                            returned tensor is a view of one of two alternating symmetric buffers: it stays
                            valid until the second next call (what the CG recurrences need), not longer.
    ``normal_op(gamma)`` -> callable for :func:`..utils.cg.cg` (tensor-op recurrences on replicated vectors).

    Inference-only: the sharded operators do not record autograd graphs and raise if an input requires grad.
    Every backprojection runs on ``base``: a base built with ``adjoint='matched'`` makes the sharded A* the
    exact transpose as well (``adjoint`` reports the base's setting).
    """

    def __init__(self, base, group=None, chunk: int = 256, reduce: str = 'nccl', multicast=None, balance: str = 'cost'):
        if reduce not in ('nccl', 'peer'):
            raise ValueError("reduce must be 'nccl' or 'peer'")
        self.reduce = reduce
        # reduce='peer': store the reduced bands once to the NVSwitch multicast address instead of once per peer
        # (None: environment variable SCD_PEER_MULTICAST=1)
        self.multicast = (os.environ.get('SCD_PEER_MULTICAST') == '1') if multicast is None else bool(multicast)
        self._peer = None
        self.base = base
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.im_shape = base.im_shape
        self.obs_shape = base.obs_shape
        # 'cost': ranges of equal projector + backprojector cost (angle_cost_ranges); 'count': equal angle counts
        if balance not in ('cost', 'count'):
            raise ValueError("balance must be 'cost' or 'count'")
        self.angle_range = angle_cost_ranges(base.angles, self.world)[self.rank] if balance == 'cost' \
            else shard_range(base.obs_shape[0], self.rank, self.world)
        self.chunk = int(chunk)
        self._comm_stream = None

    @property
    def angles(self):
        return self.base.angles

    @property
    def adjoint(self):
        return getattr(self.base, 'adjoint', 'pixel')

    # ---------------------------------------------------------------- A ----
    def trafo(self, x: Tensor) -> Tensor:
        self._no_grad_only(x, 'trafo')
        return self.base._fp(x, angle_range=self.angle_range)

    __call__ = trafo

    def gather_sinogram(self, y_local: Tensor) -> Tensor:
        """Full sinogram on every rank (rows are disjoint, so a sum all-reduce assembles them)."""
        if self.world > 1:
            y_local = y_local.clone()
            dist.all_reduce(y_local, op=dist.ReduceOp.SUM, group=self.group)
        return y_local

    # --------------------------------------------------------------- A* ----
    @staticmethod
    def _no_grad_only(t: Tensor, what: str) -> None:
        """The sharded view is inference-only: its operators bypass the autograd Functions of the wrapped
        operator (the partial results live in recycled / symmetric buffers autograd could not save), so a
        gradient through A*A would be dropped silently.  Refuse instead."""
        if torch.is_grad_enabled() and t.requires_grad:
            raise RuntimeError('AngleShardedRayTrafo.%s does not support autograd (inference-only view): call it '
                               'under torch.no_grad() or detach the input' % what)

    def _chunk_bounds(self, n: int):
        """Slice chunks ``[(lo, hi)]`` of at most ``chunk`` slices, equal in size.  The projector and backprojector like large batches more
        than the pipeline likes many chunks: 501 slices on 8 GPUs, `op` with chunks of 128 / 167 / 251 slices: 12.85 /
        13.18 / 12.67 ms (NCCL), 12.84 / 12.65 / 12.36 ms (peer-staged, multicast store) -- hence the default of 256.
        (Splitting the last chunk in two to shorten the only reduction with nothing to hide behind was also measured:
        the smaller launches cost the projector what the collective gains.)"""
        if n <= 0:
            return []
        k = -(-n // self.chunk)                        # number of chunks; sizes levelled (501 -> 251 + 250, not 256 + 245)
        return [shard_range(n, i, k) for i in range(k)]

    def _reduce_chunks(self, produce, n: int, out: Tensor) -> Tensor:
        """``out[c] = all_reduce(produce(c))`` over slice chunks, communication of chunk c overlapping the
        computation of chunk c+1 (side stream on CUDA).  ``produce(lo, hi, dst)`` writes this rank's partial of
        slices ``[lo, hi)`` into ``dst = out[lo:hi]`` (or returns another tensor, which is then copied): the
        partial is reduced IN PLACE, so the stack is written once and read once by the collective -- no
        temporary, no copy-out."""
        def make(lo, hi):
            dst = out[lo:hi]
            res = produce(lo, hi, dst)
            if res is not dst and res.data_ptr() != dst.data_ptr():
                dst.copy_(res)
            return dst
        if self.world == 1:
            for lo, hi in self._chunk_bounds(n):
                make(lo, hi)
            return out
        on_cuda = out.is_cuda
        if on_cuda and self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(device=out.device)
        pending = []
        for lo, hi in self._chunk_bounds(n):
            part = make(lo, hi)
            if on_cuda:
                ready = torch.cuda.Event()
                ready.record(torch.cuda.current_stream(out.device))
                with torch.cuda.stream(self._comm_stream):
                    self._comm_stream.wait_event(ready)
                    dist.all_reduce(part, op=dist.ReduceOp.SUM, group=self.group)
            else:
                pending.append(dist.all_reduce(part, op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        if on_cuda:
            # the caller's stream waits for the reductions: whatever touches `out` (or its memory, once freed)
            # afterwards is ordered behind the side stream's work, so no record_stream bookkeeping is needed
            torch.cuda.current_stream(out.device).wait_stream(self._comm_stream)
        else:
            for work in pending:
                work.wait()
        return out

    def _base_takes_out(self) -> bool:
        return getattr(self.base, '_out_image', None) is not None

    def trafo_adjoint(self, y: Tensor) -> Tensor:
        self._no_grad_only(y, 'trafo_adjoint')
        lead = y.shape[:-2]
        yf = y.reshape(-1, 1, *self.obs_shape)
        if self.reduce == 'peer' and self.world > 1:
            out = self._peer_state(yf.shape[0], y.device).run(
                yf.shape[0],
                lambda lo, hi, ptrs, rows: self.base._bp_banded(yf[lo:hi], self.base.adj_scale, ptrs, rows,
                                                                angle_range=self.angle_range),
                None)
            return out.clone().reshape(*lead, *self.im_shape)     # callers keep A*(y) (rhs of the sampler)
        out = torch.empty(yf.shape[0], 1, *self.im_shape, dtype=y.dtype, device=y.device)

        def produce(lo, hi, dst):
            if self._base_takes_out():
                return self.base._bp(yf[lo:hi], self.base.adj_scale, angle_range=self.angle_range, out=dst)
            return self.base._bp(yf[lo:hi], self.base.adj_scale, angle_range=self.angle_range)
        self._reduce_chunks(produce, yf.shape[0], out)
        return out.reshape(*lead, *self.im_shape)

    @staticmethod
    def _no_weights(weights) -> None:
        if weights is not None:
            raise ValueError('AngleShardedRayTrafo does not take measurement weights: run the weighted '
                             'data-consistency system on an unsharded B200RayTrafo')

    def normal_apply(self, v: Tensor, gamma: float, weights=None) -> Tensor:
        self._no_weights(weights)
        self._no_grad_only(v, 'normal_apply')
        lead = v.shape[:-2]
        vf = v.reshape(-1, 1, *self.im_shape)
        if self.reduce == 'peer' and self.world > 1:
            vf = vf.contiguous()
            out = self._peer_state(vf.shape[0], v.device).run(
                vf.shape[0],
                lambda lo, hi, ptrs, rows: self.base._normal_banded(vf[lo:hi], gamma, ptrs, rows,
                                                                    angle_range=self.angle_range),
                vf)                                   # the identity term is added by the owner's reduction
            return out.reshape(*lead, *self.im_shape)
        out = torch.empty_like(vf, memory_format=torch.contiguous_format)
        fused = getattr(self.base, 'normal_apply', None)      # B200RayTrafo: A*A without re-laying-out the sinogram
        first = self.rank == 0        # the identity term of op rides on rank 0's partial: the sum is the result

        def produce(lo, hi, dst):
            if fused is not None and self._base_takes_out():
                return fused(vf[lo:hi], gamma, angle_range=self.angle_range, add_identity=first, out=dst)
            q = self.base._fp(vf[lo:hi], angle_range=self.angle_range)
            part = self.base._bp(q, gamma * self.base.adj_scale, angle_range=self.angle_range)
            return part + vf[lo:hi] if first else part
        self._reduce_chunks(produce, vf.shape[0], out)
        return out.reshape(*lead, *self.im_shape)

    def normal_op(self, gamma: float, weights=None):
        self._no_weights(weights)
        return lambda v: self.normal_apply(v, gamma)

    def _peer_state(self, n_slices: int, device):
        if self._peer is None or self._peer.capacity < n_slices or self._peer.device != device or self._peer.m != self.chunk:
            self._peer = _PeerReduce(self, n_slices, device)
        return self._peer


def band_layout(n_rows: int, world: int):
    """Rows per band (a multiple of 32, the tallest backprojector tile) such that ``world`` bands cover
    ``n_rows`` image rows; band ``r`` = rows ``[r*band_rows, min(n_rows, (r+1)*band_rows))`` (may be empty)."""
    band_rows = -(-n_rows // world)
    band_rows = -(-band_rows // 32) * 32
    return band_rows


class _PeerReduce:
    """Symmetric buffers and the chunk pipeline of ``reduce='peer'`` (see the module docstring).

    ``stage[buf][src rank][chunk slice][band_rows][n1]`` on every rank receives the partial band of every
    rank; ``result[slice][n0][n1]`` on every rank receives the reduced bands of all owners.  Both live in
    torch symmetric memory, so every rank holds device addresses of every peer's copy."""

    NBUF = 3        # staging buffers: a rank may run two chunks ahead of the slowest owner

    def __init__(self, sh: 'AngleShardedRayTrafo', capacity: int, device):
        import torch.distributed._symmetric_memory as symm_mem
        self.sh, self.capacity, self.device = sh, int(capacity), device
        P, m = sh.world, sh.chunk
        self.m = m                                               # the staging slots are sized for this chunk
        n0, n1 = sh.im_shape
        self.band_rows = band_layout(n0, P)
        self.row_lo = min(n0, sh.rank * self.band_rows)
        self.rows = max(0, min(n0, (sh.rank + 1) * self.band_rows) - self.row_lo)
        self.slot = m * self.band_rows * n1                      # floats per (buffer, source rank)
        group = sh.group if sh.group is not None else dist.group.WORLD
        self.stage = symm_mem.empty(self.NBUF * P * self.slot, dtype=torch.float32, device=device)
        self.results = [symm_mem.empty(self.capacity * n0 * n1, dtype=torch.float32, device=device) for _ in range(2)]
        hs = symm_mem.rendezvous(self.stage, group=group)
        hr = [symm_mem.rendezvous(r, group=group) for r in self.results]
        self.stage_ptrs = [int(p) for p in hs.buffer_ptrs]       # base address of every rank's stage / results
        self.result_ptrs = [[int(p) for p in h.buffer_ptrs] for h in hr]
        self._handles = (hs, hr)
        # NVSwitch multicast address of each result buffer (0 when the box has none): the owner's reduction
        # then stores every value once and the switch replicates it, instead of one store per peer
        self.result_mc = [int(getattr(h, 'multicast_ptr', 0) or 0) for h in hr]
        # opt-in (SCD_PEER_MULTICAST=1): measured slower than per-peer stores on 2 GPUs (scalar strong.sys stores),
        # not yet measured on 8, where it divides the owner's outgoing traffic by the number of GPUs
        self.use_multicast = all(self.result_mc) and sh.multicast
        self.calls = 0
        self.flag = torch.zeros(1, device=device)
        self.comm = torch.cuda.Stream(device=device)

    def _barrier(self):
        # stream-ordered cross-rank ordering point: completes on this rank only after every rank's
        # preceding work on its side stream (hence the kernels it waited for) has completed
        dist.all_reduce(self.flag, op=dist.ReduceOp.SUM, group=self.sh.group)

    def run(self, n: int, produce, addend) -> Tensor:
        sh = self.sh
        P, m = sh.world, self.m
        n0, n1 = sh.im_shape
        main = torch.cuda.current_stream(self.device)
        stage_bytes = self.slot * 4
        which = self.calls % 2
        self.calls += 1
        result, result_ptrs, result_mc = self.results[which], self.result_ptrs[which], self.result_mc[which]
        landed = []                                              # event: barrier after chunk c's stores
        for c, (lo, hi) in enumerate(sh._chunk_bounds(n)):      # chunks of at most m slices (the staging slot size)
            buf = c % self.NBUF
            if c >= self.NBUF:
                # the owners have reduced chunk c - NBUF (their reduction precedes their barrier of chunk
                # c - NBUF + 1 in stream order): its staging buffer may be overwritten
                main.wait_event(landed[c - self.NBUF + 1])
            # my partial of band o goes to slot [buf][my rank] of owner o's stage
            ptrs = [self.stage_ptrs[o] + (buf * P + sh.rank) * stage_bytes for o in range(P)]
            produce(lo, hi, ptrs, self.band_rows)
            stored = torch.cuda.Event()
            stored.record(main)
            with torch.cuda.stream(self.comm):
                self.comm.wait_event(stored)
                self._barrier()                                  # every rank's stores of chunk c have landed
                ev = torch.cuda.Event()
                ev.record(self.comm)
                landed.append(ev)
                if self.rows > 0:
                    outs = [result_mc + lo * n0 * n1 * 4] if self.use_multicast else \
                        [result_ptrs[p] + lo * n0 * n1 * 4 for p in range(P)]
                    sh.base._band_reduce(self.stage_ptrs[sh.rank] + buf * P * stage_bytes, P, self.slot, hi - lo,
                                         self.band_rows, self.rows, self.row_lo, outs, self.device,
                                         addend=None if addend is None else addend[lo:hi],
                                         c_add=1.0 if addend is not None else 0.0, multicast=self.use_multicast)
        with torch.cuda.stream(self.comm):
            self._barrier()                                      # every owner's reduced bands have landed
        main.wait_stream(self.comm)
        # the result lives in a symmetric buffer (two alternate: valid until the second next call)
        return result[:n * n0 * n1].view(n, 1, n0, n1)
