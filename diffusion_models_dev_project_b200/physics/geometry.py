"""Host-side 2-D parallel-beam geometry (no ODL).

Restates what the reference obtains from ``odl.uniform_discr`` and
``odl.tomo.parallel_beam_geometry`` in ``SimpleTrafo.__init__``
(reference src/physics/trafo.py:18-27; rule written out in SURVEY.md §3.5 and
Appendix A):

* image domain ``[(-n)//2, n//2]^2`` with ``n x n`` unit-ish cells -- note the
  operator precedence ``-n//2 == (-n)//2``: 256 -> [-128,128], 501 -> [-251,250];
* angles: midpoints of a uniform partition of ``[0, pi)``;
* detector: ``rho`` = largest corner distance, ``n_det = 2*ceil(rho/cell)+1``
  cells on ``[-rho, rho]``.

Limited-angle and non-uniform view sets (``from_angle_range``, ``from_angles``)
keep that image domain and detector and follow ODL's ``uniform_partition`` /
``nonuniform_partition`` of the angles: every view owns an angular cell, and
A* weighs view ``i`` by its cell ``dphi * w_i`` (``dphi`` = mean cell,
``angle_weights`` = the cells relative to it, ``None`` when they are equal).
"""
from dataclasses import dataclass
from math import ceil, pi, sqrt
from typing import Optional

import numpy as np


@dataclass(frozen=True)
class ParallelBeamGeometry2D:
    n0: int
    n1: int
    x_min: float
    y_min: float
    dx: float
    angles: np.ndarray      # [n_angles] float64, radians
    n_det: int
    s_min: float
    ds: float
    angle_span: float = pi                        # total length of the angle cells (the partition's extent)
    angle_weights: Optional[np.ndarray] = None    # [n_angles] cell of each view / dphi (mean 1); None: uniform

    @property
    def n_angles(self):
        return int(self.angles.shape[0])

    @property
    def im_shape(self):
        return (self.n0, self.n1)

    @property
    def obs_shape(self):
        return (self.n_angles, self.n_det)

    @property
    def dphi(self):
        """Mean angle cell: the span of the angle partition over ``n_angles`` (``pi / n_angles`` for the
        uniform partition of [0, pi))."""
        return self.angle_span / self.n_angles

    @property
    def range_weight(self):
        """ODL cell-volume ratio c_w = dphi*ds/(dx*dx) (SURVEY.md §8b), with the mean angle cell."""
        return self.dphi * self.ds / (self.dx * self.dx)

    @property
    def view_weights(self):
        """``angle_weights`` as a float64 array (ones when ``None``)."""
        if self.angle_weights is None:
            return np.ones(self.n_angles, dtype=np.float64)
        return np.asarray(self.angle_weights, dtype=np.float64)

    @property
    def range_weights(self):
        """Per-view ODL cell-volume ratio ``c_i = dphi * w_i * ds / dx^2`` ([n_angles] float64)."""
        return self.range_weight * self.view_weights

    @staticmethod
    def _domain(im_shape):
        """Image domain and detector of ``SimpleTrafo`` (SURVEY.md §3.5): ``(n0, n1, lo, dx, n_det, rho)``."""
        n0, n1 = int(im_shape[0]), int(im_shape[1])
        lo = np.array([(-n0) // 2, (-n1) // 2], dtype=np.float64)
        hi = np.array([n0 // 2, n1 // 2], dtype=np.float64)
        cell = (hi - lo) / np.array([n0, n1], dtype=np.float64)
        if abs(cell[0] - cell[1]) > 1e-12:
            raise ValueError('only square pixels are supported (got cell sides %r)' % (cell,))
        corners = [(x, y) for x in (lo[0], hi[0]) for y in (lo[1], hi[1])]
        rho = max(sqrt(x * x + y * y) for x, y in corners)
        n_det = 2 * int(ceil(rho / float(cell.min()))) + 1
        return n0, n1, lo, float(cell[0]), n_det, rho

    @staticmethod
    def _build(im_shape, angles, angle_span=pi, angle_weights=None):
        n0, n1, lo, dx, n_det, rho = ParallelBeamGeometry2D._domain(im_shape)
        return ParallelBeamGeometry2D(
            n0=n0, n1=n1, x_min=float(lo[0]), y_min=float(lo[1]), dx=dx,
            angles=angles, n_det=n_det, s_min=-rho, ds=2.0 * rho / n_det,
            angle_span=angle_span, angle_weights=angle_weights)

    @staticmethod
    def from_im_shape(im_shape, num_angles):
        """Geometry of ``SimpleTrafo(im_shape, num_angles)``."""
        angles = (np.arange(num_angles, dtype=np.float64) + 0.5) * (pi / num_angles)
        return ParallelBeamGeometry2D._build(im_shape, angles)

    @staticmethod
    def from_angle_range(im_shape, num_angles, angle_min, angle_max):
        """``num_angles`` cell-centred views on ``[angle_min, angle_max)`` (radians): ODL's
        ``uniform_partition(angle_min, angle_max, num_angles)``, e.g. a limited-angle wedge.
        ``dphi = (angle_max - angle_min) / num_angles``; no view weights."""
        num_angles = int(num_angles)
        a0, a1 = float(angle_min), float(angle_max)
        if num_angles < 1:
            raise ValueError('from_angle_range: need at least one view (got %d)' % num_angles)
        if not (np.isfinite(a0) and np.isfinite(a1) and a1 > a0):
            raise ValueError('from_angle_range: need angle_min < angle_max (got %r, %r)' % (angle_min, angle_max))
        step = (a1 - a0) / num_angles
        angles = a0 + (np.arange(num_angles, dtype=np.float64) + 0.5) * step
        return ParallelBeamGeometry2D._build(im_shape, angles, angle_span=a1 - a0)

    @staticmethod
    def from_angles(im_shape, angles):
        """Views at the given angles (radians, any order), weighted like ODL's ``nonuniform_partition``:
        after sorting, the cell of an inner view runs from the midpoint with the previous view to the midpoint
        with the next, and each outer cell extends half the neighbouring gap past its view.  The weights are
        the cells over their mean, in the caller's order; ``None`` when the cells are all equal (to 1e-9).  A single view
        stands for the whole half turn (cell ``pi``).  Duplicate angles are rejected."""
        ang = np.array(angles, dtype=np.float64).reshape(-1)
        n = ang.size
        if n < 1:
            raise ValueError('from_angles: need at least one view')
        if not np.all(np.isfinite(ang)):
            raise ValueError('from_angles: angles must be finite')
        order = np.argsort(ang, kind='stable')
        srt = ang[order]
        if n > 1 and np.any(np.diff(srt) <= 0):
            raise ValueError('from_angles: duplicate angles')
        if n == 1:
            return ParallelBeamGeometry2D._build(im_shape, ang)
        mid = 0.5 * (srt[1:] + srt[:-1])
        edges = np.concatenate([[srt[0] - 0.5 * (srt[1] - srt[0])], mid, [srt[-1] + 0.5 * (srt[-1] - srt[-2])]])
        cells_sorted = np.diff(edges)
        span = float(edges[-1] - edges[0])
        cells = np.empty(n, dtype=np.float64)
        cells[order] = cells_sorted
        w = cells / (span / n)
        # equal up to the rounding of the angles (a uniform list): the unweighted geometry
        weights = None if np.all(np.abs(w - 1.0) <= 1e-9) else w
        return ParallelBeamGeometry2D._build(im_shape, ang, angle_span=span, angle_weights=weights)
