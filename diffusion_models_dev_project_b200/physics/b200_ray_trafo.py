"""B200RayTrafo: drop-in for the reference's ``SimpleTrafo`` backed by libscd_b200.so.

Same constructor and attributes as ``SimpleTrafo(im_shape, num_angles, impl)``
(reference src/physics/trafo.py:17-68): ``im_shape``, ``obs_shape``, ``angles``,
``trafo``/``__call__``, ``trafo_adjoint``, ``trafo_flat``, ``trafo_adjoint_flat``,
``fbp`` and ``.to(device)``.  It deliberately has no ``resize`` attribute
(``hasattr(ray_trafo, 'resize')`` probes, reference exp_utils.py:126,232).

All arithmetic runs in hand-written sm_100a kernels reached through the C ABI
(include/scd_b200.h); PyTorch only owns the buffers and the stream.  Inputs
must live on a CUDA device -- there is no CPU path.
"""
import ctypes as C
import math
import threading
from math import pi

import numpy as np
import torch
from torch import Tensor

from .. import _lib
from .base_ray_trafo import BaseRayTrafo
from .geometry import ParallelBeamGeometry2D


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _GeomHandle:
    """Owns one ``scd_geom_t*`` (device tables) for one CUDA device."""

    def __init__(self, geom: ParallelBeamGeometry2D, adj_scale: float, device: torch.device, matched: bool = False):
        lib = _lib.load()
        ang = np.ascontiguousarray(geom.angles, dtype=np.float64)
        desc = _lib.GeomDesc(
            n0=geom.n0, n1=geom.n1, x_min=geom.x_min, y_min=geom.y_min, dx=geom.dx,
            n_angles=geom.n_angles, angles=ang.ctypes.data_as(C.POINTER(C.c_double)),
            n_det=geom.n_det, s_min=geom.s_min, ds=geom.ds, adj_scale=adj_scale)
        h = C.c_void_p()
        w = None
        if geom.angle_weights is not None:
            w = np.ascontiguousarray(geom.angle_weights, dtype=np.float64)
            if w.shape != (geom.n_angles,):
                raise ValueError('angle_weights: expected shape (%d,), got %r' % (geom.n_angles, w.shape))
        wp = w.ctypes.data_as(C.POINTER(C.c_double)) if w is not None else None
        with torch.cuda.device(device):
            if matched:
                _lib.check(lib.scd_geom_create_ex(C.byref(desc), wp, _lib.SCD_GEOM_MATCHED_ADJOINT, C.byref(h)),
                           'scd_geom_create_ex')
            elif w is None:
                _lib.check(lib.scd_geom_create(C.byref(desc), C.byref(h)), 'scd_geom_create')
            else:
                _lib.check(lib.scd_geom_create_weighted(C.byref(desc), wp, C.byref(h)), 'scd_geom_create_weighted')
        self.ptr = h
        self.device = device
        self._lib = lib

    def __del__(self):
        try:
            if getattr(self, 'ptr', None):
                self._lib.scd_geom_destroy(self.ptr)
                self.ptr = None
        except Exception:  # interpreter shutdown
            pass


class _TrafoFn(torch.autograd.Function):
    """y = A x.  Backward: the unweighted transpose A^T g = A*(g)/c_w (ODL
    ``OperatorFunction`` convention, SURVEY.md §8b).  With view weights w_i, A* carries them and the
    transpose is A*(g / w)/c_w (c_w: the mean cell).  With the pixel-driven A* this pairing is off by the
    matched/unmatched gap; with ``adjoint='matched'`` (and ``adjoint_scaling='dphi'``) it is the exact
    transpose J^T g of the Joseph matrix."""

    @staticmethod
    def forward(ctx, x, rt):
        ctx.rt = rt
        return rt._fp(x)

    @staticmethod
    def backward(ctx, g):
        rt = ctx.rt
        w = rt._view_weights(g.device)
        if w is not None:
            g = g / w
        return _AdjointFn.apply(g, rt) * (1.0 / rt.geometry.range_weight), None


class _AdjointFn(torch.autograd.Function):
    """x = A* y.  Backward: c_i * (A g)_i with the per-view cell c_i = c_w * w_i."""

    @staticmethod
    def forward(ctx, y, rt):
        ctx.rt = rt
        return rt._bp(y, rt.adj_scale)

    @staticmethod
    def backward(ctx, g):
        rt = ctx.rt
        ag = _TrafoFn.apply(g, rt) * rt.geometry.range_weight
        w = rt._view_weights(g.device)
        return (ag if w is None else ag * w), None


class MeasurementWeights:
    """Per-measurement weights ``W`` of the data-consistency system (penalised weighted least squares):
    ``op(v) = v + gamma A*(W A v)``, ``rhs = xhat0 + gamma A*(W y)`` and the adaptation loss
    ``mean(W (A x - y)^2) + lambda tv(x)``.  Low-dose data weighs each bin by its photon count (the inverse of the
    variance of its log); a weight of 0 drops a measurement (dead bins, a metal trace, a view missing from one scan
    of a batch).  The view weights of the geometry stay inside A*; ``W`` comes on top of them.

    ``w``: float32 CUDA tensor of shape ``[..., n_angles, n_det]`` with at most two leading dimensions that broadcast
    to those of the observations ``[B, C]``: ``[n_angles, n_det]`` or ``[1, 1, ...]`` (one map for every sample),
    ``[B, 1, ...]`` (one per sample), ``[B, C, ...]``; finite and >= 0.  It is validated once here (one host read) and
    copied, so that every path -- the fused calls, which read a packed copy, and the tensor expressions, which read
    ``.w`` -- sees the same weights whatever later happens to the caller's tensor.  The packed copy in the projector's
    sinogram layout is made once per observation shape (and launch tuning) and cached; the fused calls then take it
    with no extra launch.  Build one object and pass it to every call: a plain tensor is validated and packed anew by
    each call it is given to."""

    def __init__(self, ray_trafo, w: Tensor):
        if not isinstance(ray_trafo, B200RayTrafo):
            raise TypeError('measurement weights need a B200RayTrafo (got %s); the angle-sharded operator does not '
                            'take them' % type(ray_trafo).__name__)
        if not isinstance(w, Tensor):
            raise TypeError('measurement weights: a torch.Tensor is required (got %s)' % type(w).__name__)
        if w.dtype != torch.float32:
            raise TypeError('measurement weights: float32 required, got %s' % w.dtype)
        obs = tuple(ray_trafo.obs_shape)
        if not 2 <= w.dim() <= 4 or tuple(w.shape[-2:]) != obs:
            raise ValueError('measurement weights: expected shape (*lead, *%r) with at most two leading dimensions, '
                             'got %r' % (obs, tuple(w.shape)))
        if not bool((torch.isfinite(w) & (w >= 0)).all()):
            raise ValueError('measurement weights must be finite and >= 0')
        if not w.is_cuda:
            raise ValueError('measurement weights must live on a CUDA device (got %s)' % w.device)
        self.ray_trafo = ray_trafo
        self.w = w.detach().clone(memory_format=torch.contiguous_format)
        self._cache = {}

    def _lead(self, lead):
        """The leading shape of the observations ``lead`` (checked: ``W`` broadcasts to it)."""
        lead = tuple(int(d) for d in lead)
        wl = tuple(self.w.shape[:-2])
        if math.prod(wl) == 1:
            return lead
        try:
            ok = torch.broadcast_shapes(wl, lead) == lead
        except RuntimeError:
            ok = False
        if not ok:
            raise ValueError('measurement weights of leading shape %r do not broadcast to observations of leading '
                             'shape %r' % (wl, lead))
        return lead

    def expanded(self, lead) -> Tensor:
        """``W`` as a contiguous ``[prod(lead), n_angles, n_det]`` tensor: the layout of observations whose leading
        dimensions are ``lead`` (cached)."""
        lead = self._lead(lead)
        key = ('user', lead)
        if key not in self._cache:
            obs, batch = tuple(self.ray_trafo.obs_shape), math.prod(lead)
            if math.prod(self.w.shape[:-2]) == 1:
                w = self.w.reshape(1, *obs).expand(batch, *obs)
            else:
                w = self.w.expand(*lead, *obs).reshape(batch, *obs)
            self._cache[key] = w.contiguous()
        return self._cache[key]

    def packed(self, lead, device) -> int:
        """Device address of ``W`` packed for observations of leading shape ``lead`` (scd_sino_weights_pack; cached
        per shape and launch tuning -- the layout depends on both; copies made under an earlier tuning are dropped)."""
        if torch.device(device) != self.w.device:
            raise ValueError('measurement weights live on %s, the operands on %s' % (self.w.device, device))
        rt = self.ray_trafo
        lead = self._lead(lead)
        key = ('il', lead, rt._tuning_epoch)
        hit = self._cache.get(key)
        if hit is None:
            for k in [k for k in self._cache if k[0] == 'il' and k[2] != rt._tuning_epoch]:
                del self._cache[k]
            w = self.expanded(lead)
            batch = w.shape[0]
            h = rt._handle(w.device)
            buf = torch.empty(int(h._lib.scd_sino_il_buffer_bytes(h.ptr, batch)) + 256, dtype=torch.uint8, device=w.device)
            ptr, _ = rt._aligned(buf)
            with torch.cuda.device(w.device):
                _lib.check(h._lib.scd_sino_weights_pack(h.ptr, w.data_ptr(), ptr, batch, _stream_ptr(w.device)),
                           'scd_sino_weights_pack')
            hit = self._cache[key] = (buf, ptr)
        return hit[1]


def as_weights(ray_trafo, weights):
    """``None``, a :class:`MeasurementWeights` of ``ray_trafo``, or a tensor to wrap in one."""
    if weights is None or isinstance(weights, MeasurementWeights):
        if weights is not None and weights.ray_trafo is not ray_trafo:
            raise ValueError('measurement weights were made for another ray transform')
        return weights
    return MeasurementWeights(ray_trafo, weights)


class NormalOp:
    """``op(v) = v + gamma * A*(A v)`` -- the closure every predictor of the
    reference builds (reference src/samplers/utils.py:188-189, 235-236, 302-303),
    as an object so that :func:`..utils.cg.cg` can recognise it and run the
    fused CUDA solve.  Calling it evaluates the operator (autograd-aware).
    With ``weights`` (a :class:`MeasurementWeights` or a tensor for one) it is ``v + gamma * A*(W A v)``."""

    def __init__(self, ray_trafo, gamma: float, weights=None):
        self.ray_trafo = ray_trafo
        self.gamma = float(gamma)
        self.weights = as_weights(ray_trafo, weights)

    def __call__(self, v: Tensor) -> Tensor:
        rt = self.ray_trafo
        if isinstance(rt, B200RayTrafo) and not (torch.is_grad_enabled() and v.requires_grad):
            return rt.normal_apply(v, self.gamma, weights=self.weights)
        av = rt(v)
        if self.weights is not None:
            av = self.weights.w * av
        return v + self.gamma * rt.trafo_adjoint(av)


class B200RayTrafo(BaseRayTrafo):
    """2-D parallel-beam ray transform on B200.

    Parameters
    ----------
    im_shape : (int, int)
    num_angles : int
    impl : str
        Accepted for signature compatibility with ``SimpleTrafo``; must be
        ``'b200'`` (or the reference's ``'odl'`` / ``'iradon'`` names, which
        select the same kernels -- there is exactly one implementation).
    adjoint_scaling : {'dphi', 'dphi/ds'}
        ``A* = adj_scale * sum_i w_i lerp(y[i], t_i(x))``; ``'dphi'`` (default) is the
        continuous weighted adjoint (kappa = 1 of SURVEY.md §8c), ``'dphi/ds'``
        the alternative kappa = 1/ds convention.  ``dphi`` is the mean angle cell and
        ``w_i`` the view weights of the geometry (1 for a uniform partition).
    adjoint : {'pixel', 'matched'}
        ``'pixel'`` (default): A* is the pixel-driven linear-interpolation backprojector (ODL / ASTRA's
        unmatched adjoint, the reference's ``SimpleTrafo``).  ``'matched'``: A* is the exact transpose of the
        Joseph projector, ``A* = (adj_scale/dphi) c_w J^T diag(w)`` with ``c_w = dphi*ds/dx^2`` (the reference's
        ``MatmulRayTrafo``), evaluated by the same kernel with a normalised hat of half-width
        ``dx max(|cos|,|sin|)/ds`` bins (``scd_geom_create_ex`` with ``SCD_GEOM_MATCHED_ADJOINT``).  Every
        backprojection of the operator uses it -- ``trafo_adjoint``, ``normal_apply``, ``cg_solve``, ``dds_step``,
        the fused adaptation objective, ``fbp`` -- so ``(I + gamma A*A)`` is symmetric positive definite and the
        gradient autograd returns through ``trafo`` is the exact transpose ``J^T g``.  ``A`` is the same either
        way.  Needs ``dx/ds < 1.5`` (every geometry ``SimpleTrafo`` derives has ``dx/ds`` just above 1).
    geometry : ParallelBeamGeometry2D, optional
        An explicit geometry (angle list and view weights, detector partition, pixel size,
        domain offset) instead of the one ``SimpleTrafo`` derives from ``(im_shape, num_angles)``;
        e.g. ``ParallelBeamGeometry2D.from_angles`` for golden-angle or randomly dropped views.
    angle_range : (float, float), optional
        ``num_angles`` cell-centred views on ``[min, max)`` radians instead of ``[0, pi)``: the
        limited-angle (missing wedge) geometry of ``ParallelBeamGeometry2D.from_angle_range``.
    """

    def __init__(self, im_shape, num_angles, impl='b200', adjoint_scaling='dphi', geometry=None, angle_range=None,
                 adjoint='pixel'):
        if impl not in ('b200', 'odl', 'iradon'):
            raise NotImplementedError(impl)
        if adjoint not in ('pixel', 'matched'):
            raise ValueError("adjoint must be 'pixel' or 'matched' (got %r)" % (adjoint,))
        self.adjoint = adjoint
        if geometry is not None and angle_range is not None:
            raise ValueError('pass either geometry or angle_range')
        if geometry is not None:
            geom = geometry
        elif angle_range is not None:
            geom = ParallelBeamGeometry2D.from_angle_range(im_shape, num_angles, *angle_range)
        else:
            geom = ParallelBeamGeometry2D.from_im_shape(im_shape, num_angles)
        if geometry is not None and (tuple(im_shape) != geom.im_shape or int(num_angles) != geom.n_angles):
            raise ValueError('geometry does not match im_shape / num_angles')
        super().__init__(im_shape=tuple(int(v) for v in im_shape), obs_shape=geom.obs_shape)
        self.geometry = geom
        if adjoint_scaling == 'dphi':
            self.adj_scale = geom.dphi
        elif adjoint_scaling == 'dphi/ds':
            self.adj_scale = geom.dphi / geom.ds
        else:
            raise ValueError(adjoint_scaling)
        self._angles = geom.angles
        self._handles = {}
        self._work = {}
        self._weights = {}
        self._tuning_epoch = 0          # bumped by set_tuning: packed measurement weights depend on the launch tuning
        self._hlock = threading.Lock()

    # ------------------------------------------------------------ plumbing ---
    @property
    def angles(self) -> np.ndarray:
        return self._angles

    def _handle(self, device: torch.device) -> _GeomHandle:
        if device.type != 'cuda':
            raise RuntimeError(
                'B200RayTrafo works on CUDA tensors only (got %s); there is no CPU fallback' % device)
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            with self._hlock:
                h = self._handles.get(idx)
                if h is None:
                    h = _GeomHandle(self.geometry, self.adj_scale, torch.device('cuda', idx),
                                    matched=self.adjoint == 'matched')
                    self._handles[idx] = h
        return h

    def _view_weights(self, device):
        """The view weights as a float32 ``[n_angles, 1]`` tensor on ``device`` (cached), or None if uniform."""
        if self.geometry.angle_weights is None:
            return None
        w = self._weights.get(device)
        if w is None:
            w = torch.as_tensor(self.geometry.view_weights, dtype=torch.float32, device=device).reshape(-1, 1)
            self._weights[device] = w
        return w

    def set_tuning(self, device, **kw):
        """Override launch heuristics (see scd_set_tuning)."""
        h = self._handle(torch.device(device))
        self._tuning_epoch += 1
        for k, v in kw.items():
            _lib.check(h._lib.scd_set_tuning(h.ptr, k.encode(), int(v)), 'scd_set_tuning')

    @staticmethod
    def _prep(t: Tensor, tail_shape, what: str) -> Tensor:
        if t.dim() < 2 or tuple(t.shape[-2:]) != tuple(tail_shape):
            raise ValueError('%s: expected trailing shape %r, got %r' % (what, tuple(tail_shape), tuple(t.shape)))
        if t.dtype != torch.float32:
            raise TypeError('%s: float32 required, got %s' % (what, t.dtype))
        return t.contiguous()

    _MAX_CACHED_BUFFERS = 24

    def _cache_put(self, key, buf: Tensor) -> None:
        """Scratch buffers are cached per (kind, device, batch size); bound the cache so that a caller
        sweeping over batch sizes does not accumulate device memory (oldest entries go first; the caching
        allocator keeps their reuse stream-ordered)."""
        while len(self._work) >= self._MAX_CACHED_BUFFERS:
            self._work.pop(next(iter(self._work)))
        self._work[key] = buf

    def workspace(self, batch: int, device: torch.device) -> Tensor:
        """Scratch for scd_cg / scd_dds_step (cached per device and batch)."""
        h = self._handle(device)
        key = (h.device.index, batch)
        w = self._work.get(key)
        if w is None:
            nbytes = int(h._lib.scd_cg_workspace_bytes(h.ptr, batch))
            w = torch.empty(nbytes + 256, dtype=torch.uint8, device=h.device)
            self._cache_put(key, w)
        return w

    def fp_scratch(self, batch: int, device: torch.device) -> Tensor:
        """Scratch for scd_fp (packed copy of the images), cached per device and batch."""
        h = self._handle(device)
        key = ('fp', h.device.index, batch)
        w = self._work.get(key)
        if w is None:
            nbytes = int(h._lib.scd_fp_scratch_bytes(h.ptr, batch))
            w = torch.empty(nbytes, dtype=torch.uint8, device=h.device)
            self._cache_put(key, w)
        return w

    def bp_scratch(self, batch: int, device: torch.device) -> Tensor:
        """Scratch for scd_bp (sample-interleaved copy of the sinograms), cached per device and batch."""
        h = self._handle(device)
        key = ('bp', h.device.index, batch)
        w = self._work.get(key)
        if w is None:
            nbytes = int(h._lib.scd_bp_scratch_bytes(h.ptr, batch))
            w = torch.empty(nbytes, dtype=torch.uint8, device=h.device)
            self._cache_put(key, w)
        return w

    @staticmethod
    def _aligned(w: Tensor):
        p = w.data_ptr()
        off = (-p) % 256
        return p + off, w.numel() - off

    # ------------------------------------------------------ raw operators ----
    def _fp(self, x: Tensor, angle_range=None) -> Tensor:
        x = self._prep(x, self.im_shape, 'trafo')
        h = self._handle(x.device)
        lead = x.shape[:-2]
        batch = int(np.prod(lead)) if len(lead) else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        if (lo, hi) == (0, self.obs_shape[0]):
            y = torch.empty(*lead, *self.obs_shape, dtype=torch.float32, device=x.device)
        else:
            y = torch.zeros(*lead, *self.obs_shape, dtype=torch.float32, device=x.device)
        scr = self.fp_scratch(batch, x.device)
        with torch.cuda.device(x.device):
            _lib.check(h._lib.scd_fp(h.ptr, x.data_ptr(), y.data_ptr(), batch, lo, hi,
                                     scr.data_ptr(), scr.numel(), _stream_ptr(x.device)), 'scd_fp')
        return y

    def _out_image(self, lead, device, out):
        """The result tensor of a backprojection: a new one, or the caller's (``out=``: a contiguous fp32 tensor
        of the result's shape, e.g. a slice of a larger stack -- the kernel then writes it in place)."""
        shape = (*lead, *self.im_shape)
        if out is None:
            return torch.empty(shape, dtype=torch.float32, device=device)
        if tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != device:
            raise ValueError('out: expected a contiguous float32 tensor of shape %r on %s' % (shape, device))
        return out

    def _bp(self, y: Tensor, scale: float, addend: Tensor = None, addend_scale: float = 0.0,
            angle_range=None, out: Tensor = None) -> Tensor:
        y = self._prep(y, self.obs_shape, 'trafo_adjoint')
        h = self._handle(y.device)
        lead = y.shape[:-2]
        batch = int(np.prod(lead)) if len(lead) else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        x = self._out_image(lead, y.device, out)
        add_ptr = None
        if addend is not None:
            addend = self._prep(addend, self.im_shape, 'addend')
            if addend.shape != x.shape:
                raise ValueError('addend shape %r != %r' % (tuple(addend.shape), tuple(x.shape)))
            add_ptr = addend.data_ptr()
        scr = self.bp_scratch(batch, y.device)
        with torch.cuda.device(y.device):
            _lib.check(h._lib.scd_bp(h.ptr, y.data_ptr(), x.data_ptr(), batch, lo, hi, float(scale),
                                     add_ptr, float(addend_scale), scr.data_ptr(), scr.numel(),
                                     _stream_ptr(y.device)), 'scd_bp')
        return x

    def _fp_il(self, x: Tensor, angle_range=None, weights=None) -> Tensor:
        """A x (``W A x`` with measurement weights) in the library's sample-interleaved sinogram layout (opaque byte
        buffer, cached per device and batch: valid until the next ``_fp_il`` of the same batch size)."""
        x = self._prep(x, self.im_shape, 'trafo')
        h = self._handle(x.device)
        batch = int(np.prod(x.shape[:-2])) if x.dim() > 2 else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        key = ('il', h.device.index, batch)
        buf = self._work.get(key)
        if buf is None:
            buf = torch.empty(int(h._lib.scd_sino_il_buffer_bytes(h.ptr, batch)) + 256, dtype=torch.uint8, device=h.device)
            self._cache_put(key, buf)
        bp, _ = self._aligned(buf)
        scr = self.fp_scratch(batch, x.device)
        wp = weights.packed(x.shape[:-2], x.device) if weights is not None else None
        with torch.cuda.device(x.device):
            _lib.check(h._lib.scd_fp_il_w(h.ptr, x.data_ptr(), bp, wp, batch, lo, hi, scr.data_ptr(), scr.numel(),
                                          _stream_ptr(x.device)), 'scd_fp_il_w')
        return buf

    def _bp_il(self, buf: Tensor, lead, scale: float, addend: Tensor = None, addend_scale: float = 0.0,
               angle_range=None, out: Tensor = None) -> Tensor:
        """Backprojection of a buffer written by :meth:`_fp_il` for the same leading shape."""
        h = self._handle(buf.device)
        batch = int(np.prod(lead)) if len(lead) else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        x = self._out_image(tuple(lead), buf.device, out)
        add_ptr = None
        if addend is not None:
            addend = self._prep(addend, self.im_shape, 'addend')
            add_ptr = addend.data_ptr()
        bp, _ = self._aligned(buf)
        with torch.cuda.device(buf.device):
            _lib.check(h._lib.scd_bp_il(h.ptr, bp, x.data_ptr(), batch, lo, hi, float(scale), add_ptr,
                                        float(addend_scale), _stream_ptr(buf.device)), 'scd_bp_il')
        return x

    # ------------------------------------------- sample-interleaved images ---
    def il_supported(self, batch: int, device) -> bool:
        """Whether batches of this size have an interleaved-image form: >= 3 samples (groups of >= 4), or a single
        sample when the image width is a multiple of 4 (its interleaved image is the reference layout itself)."""
        h = self._handle(torch.device(device))
        return int(h._lib.scd_img_il_bytes(h.ptr, int(batch))) > 0

    def _il_buffer(self, batch: int, device) -> Tensor:
        h = self._handle(device)
        n = int(h._lib.scd_img_il_bytes(h.ptr, batch))
        if n == 0:
            raise ValueError('batches of %d sample(s) have no interleaved-image form' % batch)
        buf = torch.empty(n + 256, dtype=torch.uint8, device=h.device)
        off = (-buf.data_ptr()) % 256
        return buf[off:off + n]

    def _img_il(self, x: Tensor) -> Tensor:
        """``x`` as a sample-interleaved image (opaque 256-byte aligned byte buffer, scd_img_il_pack)."""
        x = self._prep(x, self.im_shape, 'il image')
        h = self._handle(x.device)
        batch = int(np.prod(x.shape[:-2])) if x.dim() > 2 else 1
        buf = self._il_buffer(batch, x.device)
        with torch.cuda.device(x.device):
            _lib.check(h._lib.scd_img_il_pack(h.ptr, x.data_ptr(), buf.data_ptr(), batch, _stream_ptr(x.device)),
                       'scd_img_il_pack')
        return buf

    def _img_from_il(self, buf: Tensor, lead) -> Tensor:
        h = self._handle(buf.device)
        batch = int(np.prod(lead)) if len(lead) else 1
        x = torch.empty(*lead, *self.im_shape, dtype=torch.float32, device=buf.device)
        with torch.cuda.device(buf.device):
            _lib.check(h._lib.scd_img_il_unpack(h.ptr, buf.data_ptr(), x.data_ptr(), batch, _stream_ptr(buf.device)),
                       'scd_img_il_unpack')
        return x

    def _fp_ilimg(self, img_il: Tensor, batch: int, angle_range=None) -> Tensor:
        """A of an interleaved image -> interleaved sinogram: ONE launch of the projector (tensor copies straight
        from the image, no packed copy).  Returns the cached sino_il buffer of this batch size."""
        h = self._handle(img_il.device)
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        key = ('il', h.device.index, batch)
        buf = self._work.get(key)
        if buf is None:
            buf = torch.empty(int(h._lib.scd_sino_il_buffer_bytes(h.ptr, batch)) + 256, dtype=torch.uint8, device=h.device)
            self._cache_put(key, buf)
        bp, _ = self._aligned(buf)
        with torch.cuda.device(img_il.device):
            _lib.check(h._lib.scd_fp_ilimg(h.ptr, img_il.data_ptr(), bp, batch, lo, hi, _stream_ptr(img_il.device)),
                       'scd_fp_ilimg')
        return buf

    def _bp_ilimg(self, sino_il: Tensor, batch: int, scale: float, addend_il: Tensor = None, addend_scale: float = 0.0,
                  angle_range=None, out_il: Tensor = None) -> Tensor:
        """``scale * BP(sino_il) + addend_scale * addend_il`` as an interleaved image: ONE launch."""
        h = self._handle(sino_il.device)
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        out = out_il if out_il is not None else self._il_buffer(batch, sino_il.device)
        sp, _ = self._aligned(sino_il)
        with torch.cuda.device(sino_il.device):
            _lib.check(h._lib.scd_bp_ilimg(h.ptr, sp, out.data_ptr(), batch, lo, hi, float(scale),
                                           addend_il.data_ptr() if addend_il is not None else None, float(addend_scale),
                                           _stream_ptr(sino_il.device)), 'scd_bp_ilimg')
        return out

    def normal_apply(self, v: Tensor, gamma: float, angle_range=None, add_identity: bool = True,
                     out: Tensor = None, weights=None) -> Tensor:
        """``v + gamma*A*(A v)``: the projector writes the sinogram in the layout the backprojector
        stages from, the axpy is fused into the backprojector's epilogue (no grad).  ``out``: write the
        result into this tensor (may not alias ``v``).  ``weights`` (:class:`MeasurementWeights` or a tensor):
        ``v + gamma*A*(W A v)``, W applied by the projector's output phase."""
        v = self._prep(v, self.im_shape, 'normal_apply')
        q = self._fp_il(v, angle_range, weights=as_weights(self, weights))
        return self._bp_il(q, v.shape[:-2], gamma * self.adj_scale, addend=v if add_identity else None,
                           addend_scale=1.0 if add_identity else 0.0, angle_range=angle_range, out=out)

    # ---------------------------------------- banded (peer-staged) output ----
    @staticmethod
    def _ptr_array(ptrs):
        import ctypes as C
        return (C.c_void_p * len(ptrs))(*[int(p) for p in ptrs])

    def _bp_banded(self, y: Tensor, scale: float, band_ptrs, band_rows: int, angle_range=None) -> None:
        """Backprojection whose image rows ``[i*band_rows, (i+1)*band_rows)`` are stored to ``band_ptrs[i]``
        (device addresses, possibly peer memory) as dense ``[batch][band_rows][n1]`` arrays (scd_bp_banded)."""
        y = self._prep(y, self.obs_shape, 'trafo_adjoint')
        h = self._handle(y.device)
        batch = int(np.prod(y.shape[:-2])) if y.dim() > 2 else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        scr = self.bp_scratch(batch, y.device)
        with torch.cuda.device(y.device):
            _lib.check(h._lib.scd_bp_banded(h.ptr, y.data_ptr(), batch, lo, hi, float(scale), self._ptr_array(band_ptrs),
                                            len(band_ptrs), int(band_rows), scr.data_ptr(), scr.numel(),
                                            _stream_ptr(y.device)), 'scd_bp_banded')

    def _normal_banded(self, v: Tensor, gamma: float, band_ptrs, band_rows: int, angle_range=None) -> None:
        """``gamma * A*(A v)`` of this rank's angles with banded output (scd_fp_il + scd_bp_il_banded)."""
        v = self._prep(v, self.im_shape, 'normal_apply')
        h = self._handle(v.device)
        batch = int(np.prod(v.shape[:-2])) if v.dim() > 2 else 1
        lo, hi = angle_range if angle_range is not None else (0, self.obs_shape[0])
        q = self._fp_il(v, angle_range)
        qp, _ = self._aligned(q)
        with torch.cuda.device(v.device):
            _lib.check(h._lib.scd_bp_il_banded(h.ptr, qp, batch, lo, hi, float(gamma * self.adj_scale),
                                               self._ptr_array(band_ptrs), len(band_ptrs), int(band_rows),
                                               _stream_ptr(v.device)), 'scd_bp_il_banded')

    def _band_reduce(self, stage_ptr: int, n_src: int, slot_stride: int, batch: int, band_rows: int, rows: int,
                     row_lo: int, out_ptrs, device, addend: Tensor = None, c_add: float = 0.0, c_sum: float = 1.0,
                     multicast: bool = False) -> None:
        """Sum the ``n_src`` staged copies of this rank's band and store it to every ``out_ptrs[p]`` (scd_band_reduce)."""
        h = self._handle(device)
        add_ptr = None
        if addend is not None:
            addend = self._prep(addend, self.im_shape, 'addend')
            add_ptr = addend.data_ptr()
        with torch.cuda.device(device):
            _lib.check(h._lib.scd_band_reduce(int(stage_ptr), int(n_src), int(slot_stride), int(batch), int(band_rows),
                                              int(rows), self.im_shape[1], int(row_lo), self.im_shape[0],
                                              self._ptr_array(out_ptrs), len(out_ptrs), int(bool(multicast)), add_ptr, float(c_add),
                                              float(c_sum), _stream_ptr(device)), 'scd_band_reduce')

    # --------------------------------------------------- reference interface --
    def trafo(self, x: Tensor) -> Tensor:
        if torch.is_grad_enabled() and x.requires_grad:
            return _TrafoFn.apply(x, self)
        return self._fp(x)

    def trafo_adjoint(self, observation: Tensor) -> Tensor:
        if torch.is_grad_enabled() and observation.requires_grad:
            return _AdjointFn.apply(observation, self)
        return self._bp(observation, self.adj_scale)

    trafo_flat = BaseRayTrafo._trafo_flat_via_trafo
    trafo_adjoint_flat = BaseRayTrafo._trafo_adjoint_flat_via_trafo_adjoint

    def normal_op(self, gamma: float, weights=None) -> NormalOp:
        return NormalOp(self, gamma, weights)

    # ------------------------------------------------------------- solvers ---
    def cg_solve(self, x0: Tensor, rhs: Tensor, gamma: float, n_iter: int, weights=None) -> Tensor:
        """Fused batched CG on ``(I + gamma A*A) x = rhs`` from ``x0`` (no grad).
        Same recurrences as the reference's ``cg`` (src/utils/cg.py:11-39).  ``weights``: the system
        ``(I + gamma A*WA)`` (:class:`MeasurementWeights`); ``rhs`` is the caller's, e.g. ``x0 + gamma A*(W y)``."""
        x0 = self._prep(x0, self.im_shape, 'cg x')
        rhs = self._prep(rhs, self.im_shape, 'cg rhs')
        if rhs.shape != x0.shape:
            raise ValueError('cg: x %r and rhs %r differ in shape' % (tuple(x0.shape), tuple(rhs.shape)))
        if rhs.device != x0.device:
            raise ValueError('cg: x and rhs live on different devices')
        h = self._handle(x0.device)
        batch = int(np.prod(x0.shape[:-2])) if x0.dim() > 2 else 1
        weights = as_weights(self, weights)
        wil = weights.packed(x0.shape[:-2], x0.device) if weights is not None else None
        x = x0.clone()
        w = self.workspace(batch, x0.device)
        wp, wn = self._aligned(w)
        with torch.cuda.device(x0.device):
            _lib.check(h._lib.scd_cg_w(h.ptr, x.data_ptr(), rhs.data_ptr(), wil, float(gamma), int(n_iter), batch,
                                       wp, wn, _stream_ptr(x0.device)), 'scd_cg_w')
        return x

    def dds_step(self, x: Tensor, s: Tensor, atb: Tensor, eps: Tensor, t: Tensor, t_prev: Tensor,
                 abar: Tensor, gamma: float, eta: float, n_iter: int, weights=None):
        """Tweedie -> rhs -> CG -> DDIM in one library call; returns ``(x_next, xhat0)``
        (reference src/samplers/utils.py:195-218).  ``weights``: CG on ``(I + gamma A*WA)``
        (:class:`MeasurementWeights`); ``atb`` is then ``A*(W y)``."""
        x = self._prep(x, self.im_shape, 'dds x')
        s = self._prep(s, self.im_shape, 'dds s')
        atb = self._prep(atb, self.im_shape, 'dds rhs')
        eps = self._prep(eps, self.im_shape, 'dds eps')
        for name, v in (('s', s), ('eps', eps)):
            if v.shape != x.shape:
                raise ValueError('dds_step: %s shape %r != x shape %r' % (name, tuple(v.shape), tuple(x.shape)))
        batch = int(np.prod(x.shape[:-2])) if x.dim() > 2 else 1
        if atb.shape != x.shape:
            atb = atb.expand_as(x).contiguous()
        t = t.to(device=x.device, dtype=torch.float32).contiguous()
        t_prev = t_prev.to(device=x.device, dtype=torch.float32).contiguous()
        if t.numel() != batch or t_prev.numel() != batch:
            raise ValueError('dds_step: time steps must have one entry per sample')
        h = self._handle(x.device)
        weights = as_weights(self, weights)
        wil = weights.packed(x.shape[:-2], x.device) if weights is not None else None
        x_next = torch.empty_like(x)
        xhat0 = torch.empty_like(x)
        w = self.workspace(batch, x.device)
        wp, wn = self._aligned(w)
        with torch.cuda.device(x.device):
            _lib.check(h._lib.scd_dds_step_w(
                h.ptr, x.data_ptr(), s.data_ptr(), atb.data_ptr(), wil, eps.data_ptr(), t.data_ptr(),
                t_prev.data_ptr(), abar.data_ptr(), int(abar.numel()), float(gamma), float(eta), int(n_iter),
                x_next.data_ptr(), xhat0.data_ptr(), batch, wp, wn, _stream_ptr(x.device)), 'scd_dds_step_w')
        return x_next, xhat0

    # ----------------------------------------------------------------- fbp ---
    def ramp_filter(self, observation: Tensor) -> Tensor:
        """Detector-axis ramp filter of :meth:`fbp` (``scd_ramp_filter``: direct convolution with the
        band-limited ramp of Kak & Slaney in shared memory, divided by the detector cell size)."""
        y = self._prep(observation, self.obs_shape, 'fbp')
        h = self._handle(y.device)
        batch = int(np.prod(y.shape[:-2])) if y.dim() > 2 else 1
        out = torch.empty_like(y)
        with torch.cuda.device(y.device):
            _lib.check(h._lib.scd_ramp_filter(h.ptr, y.data_ptr(), out.data_ptr(), batch, _stream_ptr(y.device)),
                       'scd_ramp_filter')
        return out

    def fbp(self, observation: Tensor) -> Tensor:
        """Ram-Lak filtered back-projection: ``fbp(A x) ~ x``.

        Counterpart of ``SimpleTrafo.fbp`` (reference src/physics/trafo.py:34,42,67).  The filter is the
        recipe of the reference's ``filter_sinogram`` (src/physics/utils.py:11-33: rows zero-padded to a power
        of two >= 2 N_s, "ramp" Fourier filter ``2 Re FFT(f)`` of the Kak-Slaney kernel, scale
        ``pi/(2 N_theta)``), evaluated as the equivalent linear convolution by ``scd_ramp_filter``; the
        recipe's constants are split as ``2 * pi/(2 N_theta) = dphi`` (the weight of the pixel-driven
        backprojector) times ``1/ds`` (the recipe assumes a unit detector cell; ours is ``ds``).

        On a weighted geometry the backprojector sums view ``i`` with ``dphi * w_i``, its angular cell: the
        FBP quadrature of a non-uniform view set.  On a wedge the result is the truncated FBP -- the inverse
        Radon formula restricted to the measured angles -- not a limited-angle reconstruction: the missing
        wedge stays missing (streaks and lost edges along it).

        On a matched operator (``adjoint='matched'``) the filtered rows are backprojected with the normalised
        hat of the matched A*, i.e. by ``c_w J^T``: the result is ``(dphi/dx^2) J^T diag(w) (ds * ramp_filter(y))``,
        which on the uniform partition of [0, pi) is ``J^T filter_sinogram(y) / dx^2`` with the reference's
        ``filter_sinogram``."""
        return self._bp(self.ramp_filter(observation), self.geometry.dphi)
