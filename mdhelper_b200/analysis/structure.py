"""
Bulk structural analysis on B200
================================

GPU drop-ins for the two classes of ``mdhelper.analysis.structure`` that sit on
the per-frame hot path (reference: ``/root/reference/src/mdhelper/analysis/
structure.py``):

* :func:`radial_histogram` -- seam #1, ``structure.py:32-104``.
* :class:`RadialDistributionFunction` -- ``structure.py:444-1032``.
* :class:`StructureFactor` -- ``structure.py:1034-1550``.
* :class:`IntermediateScatteringFunction` -- ``structure.py:1552-2127`` (the first
  "next" row of the scope table: it reuses the S(q) kernels for ``rho(q, t)`` and
  for the displacement sums of the incoherent part).

Constructors, ``run(start, stop, step, frames)`` and ``results.*`` follow the
reference.  The distance / binning loop and the Fourier sums run in
``libmdh_b200.so``; everything that is O(n_bins) or O(N_q) (edges,
normalisation, unique-|q| grouping, sorting) stays in numpy so that identical
counts give identical ``results.rdf``.
"""

from __future__ import annotations

from itertools import combinations_with_replacement
from typing import Union

import numpy as np

from . import _postprocess
from ._binning import squared_thresholds
from ._triclinic import box_volume, is_orthorhombic, triclinic_vectors
from ._postprocess import (calculate_coordination_numbers,  # noqa: F401  (re-exported,
                           calculate_structure_factor,       # as in the reference module)
                           radial_fourier_transform,
                           zeroth_order_hankel_transform)
from .base import FrameFeeder, GpuAnalysisBase, all_reduce_sum, world

_GROUPINGS_RDF = {"atoms", "residues", "segments"}
_GROUPINGS_SSF = {"atoms", "residues"}


def _cell_matrices(dims: np.ndarray) -> np.ndarray:
    """``[n, 3, 3]`` float32 cell matrices of the triclinic frames ``dims`` (``[n, 6]``)."""
    cells = np.stack([triclinic_vectors(d) for d in np.atleast_2d(dims)])
    if not np.all(cells[:, [0, 1, 2], [0, 1, 2]] > 0):
        raise ValueError("Invalid unit cell dimensions.")
    return cells


def _record(batch):
    import torch
    batch.event = torch.cuda.Event()
    batch.event.record()


def _centers_of_mass(group, grouping: str, positions: np.ndarray) -> np.ndarray:
    """
    Centres of mass of the residues / segments of ``group`` (host-side helper;
    reference: ``algorithm/molecule.py:15-310`` as used at
    ``structure.py:753-756``).  float64 mass-weighted mean of the float32
    coordinates.
    """
    key = group.resindices if grouping == "residues" else group.segindices
    _, inv = np.unique(key, return_inverse=True)
    m = np.asarray(group.masses, dtype=np.float64)
    tot = np.bincount(inv, weights=m)
    com = np.empty((tot.size, 3))
    for k in range(3):
        com[:, k] = np.bincount(inv, weights=m * positions[:, k]) / tot
    return com


def _com_plan(group, grouping: str):
    """
    ``(starts, masses)`` for the device centre-of-mass kernel if the entities of
    ``group`` are consecutive runs of a contiguous atom range (the usual topology
    order), else ``None`` (the host helper is used).  ``grouping="atoms"`` gives the
    identity plan (one atom per entity, unit masses: ``(1 * x) / 1`` is exact).
    """
    ix = np.asarray(group.ix)
    if ix.size == 0 or ix[-1] - ix[0] + 1 != ix.size or np.any(np.diff(ix) != 1):
        return None
    if grouping == "atoms":
        return np.arange(ix.size + 1, dtype=np.int64), np.ones(ix.size)
    key = np.asarray(group.resindices if grouping == "residues" else group.segindices)
    change = np.flatnonzero(np.diff(key) != 0) + 1
    starts = np.concatenate(([0], change, [key.size])).astype(np.int64)
    if len(np.unique(key)) != len(starts) - 1:      # an entity split into several runs
        return None
    return starts, np.asarray(group.masses, dtype=np.float64)


def _n_entities(group, grouping: str) -> int:
    return int(getattr(group, f"n_{grouping}"))


def radial_histogram(
        pos1: np.ndarray, pos2: np.ndarray, n_bins: int, range: tuple,
        dims: tuple, *, exclusion: tuple = None, mode: str = "auto",
        hist: str = "auto", arith: str = "auto", wrap: str = "auto",
        device: int = None, stats: dict = None) -> np.ndarray:
    """
    Computes the radial histogram of distances between particles of the same
    type or two different types (GPU version of ``structure.py:32-104``).

    Parameters
    ----------
    pos1, pos2 : `numpy.ndarray`
        Positions of the two groups, shapes :math:`(N_1,\\,3)` and
        :math:`(N_2,\\,3)` (a single ``(3,)`` coordinate is one particle).
        Converted to float32, as ``capped_distance`` does.
    n_bins : `int`
        Number of histogram bins.
    range : array-like
        Range of radii values, shape ``(2,)``.
    dims : array-like
        System dimensions and orthogonality, shape ``(6,)``.
    exclusion : array-like, keyword-only, optional
        Tiles to exclude: pairs with ``i // exclusion[0] == j // exclusion[1]``
        are dropped.
    mode, hist : `str`, keyword-only
        Kernel selectors (``"auto"``, ``"allpairs"``, ``"cells"``;
        ``"auto"``, ``"warp_atomic"``, ``"lane_private"``).  Counts do not
        depend on them.
    arith : `str`, keyword-only
        ``"auto"``: fp32 filter in front of the reference's fp64 arithmetic
        (pairs provably inside a bin are binned from fp32, all others are
        re-evaluated exactly); ``"off"``: fp64 for every pair; ``"audit"``:
        filter plus a full exact comparison (test aid).  Counts do not depend
        on it either.  On triclinic cells it applies to the all-pairs kernel and
        to the cell list.  All pairs: frames whose ``range[1]`` plus the error
        bound does not fit inside half the shortest of a_x, b_y, c_z (or with
        non-finite coordinates) are declined and take the 27-image fp64
        arithmetic.  Cell list: frames with a coordinate far outside the cell,
        with non-finite coordinates, or whose cell gives a bound that is not
        small against a bin are declined and take the cell list's fp64
        arithmetic.
    wrap : `str`, keyword-only
        Coordinates outside the cell: ``"auto"`` follows the reference --
        ``capped_distance`` moves both coordinate sets into the cell in float32 before
        taking differences whenever it picks its grid search (both groups have at least
        10 particles and ``n1 * n2 >= 1e8`` or ``range[1] <= 0.3 *`` the shortest cell
        edge) and takes the differences of the coordinates as given otherwise;
        ``"never"`` / ``"always"`` force one of the two.  No effect on coordinates inside
        ``[0, L)``.
    stats : `dict`, keyword-only, optional
        If given, receives the filter statistics of the call.

    Returns
    -------
    histogram : `numpy.ndarray`
        Radial histogram, int64, shape :math:`(N_\\mathrm{bins},)`.
    """
    from .._lib import Context
    p1 = np.ascontiguousarray(np.atleast_2d(np.asarray(pos1)), dtype=np.float32)
    p2 = np.ascontiguousarray(np.atleast_2d(np.asarray(pos2)), dtype=np.float32)
    if dims is None:
        raise ValueError("Trajectory does not contain system dimension "
                         "information.")
    dims = np.asarray(dims, dtype=np.float32)
    ortho = bool(is_orthorhombic(dims)[0])
    import torch
    dev = torch.cuda.current_device() if device is None else device
    ctx = Context(dev)
    try:
        ctx.rdf_set_filter(arith)
        ctx.rdf_set_prewrap(wrap)
        # the same array twice: the kernels may use the pair symmetry (same counts) --
        # unless the exclusion blocks differ, i // e0 == j // e1 is not symmetric then
        same = pos2 is pos1 and (exclusion is None or exclusion[0] == exclusion[1])
        ctx.rdf_configure(len(p1), len(p2), same,
                          squared_thresholds(n_bins, range), range[0], range[1],
                          exclusion=exclusion, mode=mode, hist=hist)
        if ortho:
            ctx.rdf_accumulate(p1, 3 * len(p1), p2, 3 * len(p2), dims[None, :3], 1)
        else:
            ctx.rdf_accumulate_triclinic(p1, 3 * len(p1), p2, 3 * len(p2),
                                         _cell_matrices(dims[None, :]), 1)
        out = ctx.rdf_fetch()
        if stats is not None:
            stats.update(ctx.rdf_filter_stats())
        return out
    finally:
        ctx.close()


class RadialDistributionFunction(GpuAnalysisBase):
    r"""
    Radial distribution function :math:`g_{ij}(r)` between two groups for two-
    and three-dimensional periodic systems, computed on the GPU.

    Same constructor and results as the reference class
    (``structure.py:444-1032``); the differences are listed under *Notes*.

    Parameters
    ----------
    ag1, ag2 : atom groups
        First and (optionally) second group; ``ag2=None`` means ``ag1``.
    n_bins : `int`, default: :code:`201`
        Number of histogram bins.
    range : array-like, default: :code:`(0.0, 15.0)`
        Range of radii values.
    drop_axis : `int` or `str`, keyword-only, optional
        Axis to ignore for two-dimensional systems (``0/1/2`` or ``"x"/"y"/"z"``).
    norm : `str`, keyword-only, default: :code:`"rdf"`
        ``"rdf"``, ``"density"`` or :code:`None` (raw counts).
    exclusion : array-like, keyword-only, optional
        Tiles to exclude from the interparticle distances, e.g. ``(1, 1)``.
    groupings : `str` or array-like, keyword-only, default: :code:`"atoms"`
        ``"atoms"``, ``"residues"`` or ``"segments"`` (centres of mass, computed
        on the host).
    reduced : `bool`, keyword-only, default: :code:`False`
        Whether the data is in reduced units.
    n_batches : `int`, keyword-only, optional
        Accepted for compatibility and ignored: the GPU kernels never
        materialise the pair list, so the range does not need to be split.
    parallel : `bool`, keyword-only, default: :code:`False`
        Accepted for compatibility; frames are sharded over GPUs whenever
        ``torch.distributed`` is initialised.
    verbose : `bool`, keyword-only, default: :code:`True`
        Determines whether progress is logged.
    mode, hist, arith, wrap : `str`, keyword-only
        Kernel selectors and the treatment of coordinates outside the cell, see
        :func:`radial_histogram`.
    host_com : `bool`, keyword-only, default: :code:`False`
        Compute centres of mass on the host even where the device kernel applies
        (entities that are consecutive atom runs); the results are identical.

    Attributes
    ----------
    results.edges, results.bins, results.counts, results.rdf
        As in the reference; ``results.counts`` is int64 and bit-exact.

    Notes
    -----
    * ``n_batches`` has no effect (the reference documents that its batched
      mode can be off by a few counts, ``structure.py:601-607``; the GPU result
      is the unbatched one).
    * Triclinic cells run through separate kernels (coordinates wrapped into the cell,
      shortest of the 27 images per pair): ``mode="allpairs"`` evaluates all 27 images of
      every pair, ``mode="cells"`` a cell list in fractional coordinates that evaluates
      the one image per candidate that can be in range (same counts; every perpendicular
      width of the cell must hold 3 cells of ``range[1]`` plus a small margin), and
      ``"auto"`` takes the cell list for cut-off runs on large systems.
    * ``drop_axis`` works with every cell shape and ``mode``, as in the reference: the
      coordinate is zeroed, the dropped edge is widened to the longest one (a triclinic
      cell keeps its angles) and the accumulated area is the product of the two other
      edges -- for a hexagonal cell ``a * b``, not ``a * b * sin(gamma)``, which is what
      the reference computes.  The cell list takes a dropped axis with one cell along it
      (orthorhombic cells: any axis; triclinic cells: ``drop_axis=2`` only, with
      ``c_z`` at least ``range[1]`` plus a small margin).  ``mode="cells"`` raises
      ``ValueError`` for a triclinic cell with ``drop_axis`` 0 or 1, which
      ``"auto"`` runs through all pairs.
    """

    def __init__(
            self, ag1, ag2=None, n_bins: int = 201,
            range: tuple = (0.0, 15.0), *, drop_axis: Union[int, str] = None,
            norm: str = "rdf", exclusion: tuple = None,
            groupings: Union[str, tuple] = "atoms", reduced: bool = False,
            n_batches: int = None, parallel: bool = False,
            verbose: bool = True, mode: str = "auto", hist: str = "auto",
            arith: str = "auto", wrap: str = "auto", host_com: bool = False,
            **kwargs) -> None:

        self.ag1 = ag1
        self.ag2 = ag1 if ag2 is None else ag2
        self.universe = self.ag1.universe
        if self.universe.dimensions is None:
            raise ValueError("Trajectory does not contain system "
                             "dimension information.")

        super().__init__(self.universe.trajectory, verbose, **kwargs)
        self._parallel = parallel

        if isinstance(groupings, str):
            if groupings not in _GROUPINGS_RDF:
                emsg = (f"Invalid grouping '{groupings}'. The options are "
                        "'atoms', 'residues', and 'segments'.")
                raise ValueError(emsg)
            self._groupings = 2 * [groupings]
        else:
            for g in groupings:
                if g not in _GROUPINGS_RDF:
                    emsg = (f"Invalid grouping '{g}'. The options are "
                            "'atoms', 'residues', and 'segments'.")
                    raise ValueError(emsg)
            self._groupings = (2 * list(groupings) if len(groupings) == 1
                               else list(groupings))

        self._drop_axis = (ord(drop_axis) - 120 if isinstance(drop_axis, str)
                           else drop_axis)
        if self._drop_axis not in {0, 1, 2, None}:
            raise ValueError("Invalid axis to drop.")

        self._n_bins = n_bins
        self._range = range
        self._norm = norm
        self._exclusion = exclusion
        self._reduced = reduced
        self._n_batches = n_batches
        self._verbose = verbose
        self._mode = mode
        self._hist = hist
        self._arith = arith
        self._wrap = wrap
        self._host_com = bool(host_com)
        self._com = None

    def _prepare(self) -> None:
        # reference: structure.py:734-748
        self.results.edges = np.linspace(*self._range, self._n_bins + 1)
        self.results.bins = (self.results.edges[:-1]
                             + self.results.edges[1:]) / 2
        self.results.counts = np.zeros(self._n_bins, dtype=int)
        self.results.units = {"results.bins": "angstrom",
                              "results.edges": "angstrom"}
        self._area_or_volume = 0.0

    def _begin(self, frames: np.ndarray):
        """Configures the context; returns ``(index_sets, positions_fn,
        bytes_per_frame)`` for the frame feeder."""
        ctx = self._context()
        n1 = _n_entities(self.ag1, self._groupings[0])
        n2 = _n_entities(self.ag2, self._groupings[1])
        # one packed copy and the pair symmetry are only valid when the exclusion test
        # i // e0 == j // e1 (structure.py:100-102) is symmetric as well
        same = (self.ag1 is self.ag2
                or np.array_equal(self.ag1.ix, self.ag2.ix)) \
            and self._groupings[0] == self._groupings[1] \
            and (not self._exclusion or self._exclusion[0] == self._exclusion[1])
        self._same = same
        ctx.rdf_set_filter(self._arith)
        ctx.rdf_set_prewrap(self._wrap)
        if getattr(self, "_thresholds", None) is None:   # fixed per instance
            self._thresholds = squared_thresholds(self._n_bins, self._range)
        ctx.rdf_configure(
            n1, n2, same, self._thresholds,
            self._range[0], self._range[1], exclusion=self._exclusion,
            drop_axis=self._drop_axis, mode=self._mode, hist=self._hist
        )
        self._kernel_ms = 0.0
        atoms_only = self._groupings[0] == self._groupings[1] == "atoms"
        sets = [self.ag1.ix] if same else [self.ag1.ix, self.ag2.ix]
        positions_fn = None
        self._com = None
        if not atoms_only:
            groups = [self.ag1] if same else [self.ag1, self.ag2]
            grps = self._groupings[:len(groups)]
            plans = [_com_plan(g, gr) for g, gr in zip(groups, grps)]
            if all(p is not None for p in plans) and not self._host_com:
                # centres of mass on the device: the feeder hands over the raw atoms
                for slot, (starts, masses) in enumerate(plans):
                    ctx.com_configure(slot, starts, masses)
                self._com = [len(p[0]) - 1 for p in plans]
                return [g.ix for g in groups], None, 12 * sum(g.n_atoms for g in groups)

            def positions_fn(ts, groups=groups, grps=grps):
                return [ts.positions[g.ix] if gr == "atoms"
                        else _centers_of_mass(g, gr, ts.positions[g.ix])
                        for g, gr in zip(groups, grps)]
            sets = [np.arange(n1)] if same else [np.arange(n1), np.arange(n2)]
        return sets, positions_fn, 12 * (n1 + n2)

    def _consume(self, batch, device: bool = False) -> None:
        """One batch of frames (host or device pointers) into the accumulators."""
        ortho = is_orthorhombic(batch.dims)
        box = batch.dims[:, :3].copy()
        if self._drop_axis is None:
            # ts.volume: float64 product of the float32 edges (times the angular factor
            # of a triclinic cell)
            for d, o, v in zip(batch.dims, ortho, box.astype(np.float64).prod(axis=1)):
                self._area_or_volume += v if o else box_volume(d)
        else:
            # reference: structure.py:764-770 -- the dropped edge widened to the longest one,
            # the angles kept; the area is the product of the two other edges for every cell
            # shape (a * b for a hexagonal cell, not a * b * sin(gamma): as the reference)
            box[:, self._drop_axis] = box.max(axis=1)
            keep = [k for k in (0, 1, 2) if k != self._drop_axis]
            for v in box[:, keep].astype(np.float64).prod(axis=1):
                self._area_or_volume += v
        dims = batch.dims.copy()
        dims[:, :3] = box
        same = self._same
        ptrs, strides = batch.ptrs, batch.strides
        if self._com is not None:
            # raw atoms -> centres of mass on the device (com.cu); the kernels that
            # read `outs` are queued on torch's current stream, so the allocator cannot
            # recycle them early
            import torch
            outs = [torch.empty((batch.n_frames, n, 3), dtype=torch.float32,
                                device=f"cuda:{self._device}") for n in self._com]
            for slot, out in enumerate(outs):
                self._ctx.com_reduce(slot, ptrs[slot], strides[slot], batch.n_frames,
                                     out, 3 * self._com[slot], device=device)
            ptrs = [o.data_ptr() for o in outs]
            strides = [3 * n for n in self._com]
            device = True
        # runs of frames with the same kind of cell (a trajectory is normally all of one)
        f0 = 0
        while f0 < batch.n_frames:
            f1 = f0 + 1
            while f1 < batch.n_frames and ortho[f1] == ortho[f0]:
                f1 += 1
            p1 = ptrs[0] + 4 * strides[0] * f0
            p2 = None if same else ptrs[1] + 4 * strides[1] * f0
            s2 = 0 if same else strides[1]
            if ortho[f0]:
                self._ctx.rdf_accumulate(p1, strides[0], p2, s2, box[f0:f1], f1 - f0,
                                         device=device, keepalive=batch.keepalive)
            else:
                # triclinic: coordinates wrapped into the cell (of the widened dimensions
                # with drop_axis), shortest of 27 images
                self._ctx.rdf_accumulate_triclinic(
                    p1, strides[0], p1 if same else p2, strides[0] if same else s2,
                    _cell_matrices(dims[f0:f1]), f1 - f0, device=device,
                    keepalive=batch.keepalive)
            f0 = f1
        _record(batch)

    def _finish(self) -> None:
        ctx = self._ctx
        self._local_counts = ctx.rdf_fetch()
        self._pair_evaluations = ctx.rdf_pair_evaluations()
        self._filter_stats = ctx.rdf_filter_stats()

    def _conclude(self) -> None:
        # one all-reduce: counts (exact) and the accumulated volume
        counts = all_reduce_sum(self._local_counts, self._device)
        vol = all_reduce_sum(np.array([self._area_or_volume]), self._device)[0]
        self.results.counts[:] = counts
        self._area_or_volume = float(vol)

        # normalisation, reference: structure.py:844-862
        norm = self.n_frames
        if self._norm is not None:
            if self._drop_axis is None:
                norm = norm * (4 * np.pi * np.diff(self.results.edges ** 3) / 3)
            else:
                norm = norm * (np.pi * np.diff(self.results.edges ** 2))
            if self._norm == "rdf":
                _N2 = _n_entities(self.ag2, self._groupings[1])
                if self._exclusion:
                    _N2 -= self._exclusion[1]
                norm = norm * (_n_entities(self.ag1, self._groupings[0]) * _N2
                               * self.n_frames / self._area_or_volume)
        self.results.rdf = self.results.counts / norm

    def _get_rdf(self) -> np.ndarray:
        """
        Returns the radial distribution function whatever ``norm`` was
        (reference: ``structure.py:864-891``).
        """
        if self._norm == "rdf":
            return self.results.rdf
        _N2 = _n_entities(self.ag2, self._groupings[1])
        if self._exclusion:
            _N2 -= self._exclusion[1]
        if self._drop_axis is None:
            norm = 4 * np.diff(self.results.edges ** 3) / 3
        else:
            norm = np.diff(self.results.edges ** 2)
        return self._area_or_volume * self.results.counts / (
            np.pi * self.n_frames ** 2 * _N2 * norm
            * _n_entities(self.ag1, self._groupings[0])
        )

    def calculate_coordination_numbers(self, rho: float, *, n_coord_nums: int = 2,
                                       threshold: float = 0.1) -> None:
        """
        Coordination numbers from the minima of :math:`g(r)` into
        ``results.coordination_numbers`` (reference: ``structure.py:893-923``).

        Parameters
        ----------
        rho : `float`
            Number density of the surrounding species.
        n_coord_nums : `int`, keyword-only, default: :code:`2`
            Number of coordination numbers to calculate.
        threshold : `float`, keyword-only, default: :code:`0.1`
            Minimum :math:`g(r)` a local minimum must have to count.
        """
        self.results.coordination_numbers = \
            _postprocess.calculate_coordination_numbers(
                self.results.bins, self._get_rdf(), rho, n_coord_nums=n_coord_nums,
                n_dims=2 + (self._drop_axis is None), threshold=threshold)

    def calculate_pmf(self, temperature: float) -> None:
        """
        Potential of mean force :math:`-k_\\mathrm{B}T\\ln g(r)` into ``results.pmf``
        (kJ/mol, or reduced units when ``reduced=True``; reference:
        ``structure.py:925-959``).  ``temperature`` is a plain number (kelvin).
        """
        self.results.units["results.pmf"] = "kilojoule / mole"
        kBT = _postprocess.thermal_energy(temperature, self._reduced)
        with np.errstate(divide="ignore"):
            self.results.pmf = -kBT * np.log(self._get_rdf())

    def calculate_structure_factor(self, rho: float, x_i: float = None,
                                   x_j: float = None, q: np.ndarray = None, *,
                                   q_lower: float = None, q_upper: float = None,
                                   n_q: int = 1_000, formalism: str = "FZ") -> None:
        """
        (Partial) static structure factor from :math:`g(r)` by a radial Fourier
        (3-D) or Hankel (2-D) transform into ``results.wavenumbers`` and
        ``results.ssf`` (reference: ``structure.py:961-1031``).
        """
        equal = (self.ag1 is self.ag2
                 or np.array_equal(self.ag1.ix, self.ag2.ix))
        self.results.wavenumbers, self.results.ssf = \
            _postprocess.calculate_structure_factor(
                self.results.bins, self._get_rdf(), equal, rho, x_i, x_j, q=q,
                q_lower=q_lower, q_upper=q_upper, n_q=n_q,
                n_dims=2 + (self._drop_axis is None), formalism=formalism)


def _grid_indices(n_points: int) -> np.ndarray:
    """``[n_points^3, 3]`` indices of the first-octant grid in the reference's
    ``np.meshgrid`` 'xy' order: row (i, j, k) holds (j, i, k)."""
    idx = np.arange(n_points)
    ii, jj, kk = np.meshgrid(idx, idx, idx, indexing="ij")
    return np.stack((jj, ii, kk), axis=-1).reshape(-1, 3)


def _lattice_indices(wavevectors: np.ndarray, dimensions) -> tuple:
    """
    If every wavevector is a non-negative integer multiple of the reciprocal
    lattice basis ``b_k = 2 pi / L_k``, returns ``(n, b)``; else ``(None, None)``.
    """
    if dimensions is None:
        return None, None
    b = 2 * np.pi / np.asarray(dimensions, dtype=np.float64)
    n = np.rint(wavevectors / b)
    if (n < 0).any() or (n > 1023).any():
        return None, None
    if not np.allclose(n * b, wavevectors, rtol=1e-12, atol=1e-12 * b.max()):
        return None, None
    n = n.astype(np.int32)
    if len(np.unique(n, axis=0)) != len(n):
        return None, None
    return n, b


class StructureFactor(GpuAnalysisBase):
    r"""
    Static (or partial) structure factor by direct summation,

    .. math::

       S(\mathbf{q})=\frac{1}{N}\left\langle\left|\sum_{j=1}^N
       \exp(i\mathbf{q}\cdot\mathbf{r}_j)\right|^2\right\rangle,

    on the first-octant reciprocal-lattice grid of the box (or on user supplied
    wavevectors), computed on the GPU.  Same constructor and results as the
    reference class (``structure.py:1034-1550``).

    Parameters
    ----------
    groups : atom group or sequence of atom groups
    groupings : `str` or sequence, default: :code:`"atoms"`
        ``"atoms"`` or ``"residues"`` (centres of mass, computed on the host).
    mode : `str`, keyword-only, optional
        :code:`None` (all particles together), ``"pair"`` or ``"partial"``.
    form : `str`, keyword-only, default: :code:`"exp"`
        ``"exp"`` or ``"trig"``; both are served by the same kernels
        (``|sum exp|^2 == (sum cos)^2 + (sum sin)^2``).
    dimensions, n_points, n_surfaces, n_surface_points, q_max, wavevectors,
    sort, unique
        As in the reference (``structure.py:1366-1416``).
    reciprocal : `str`, keyword-only, default: :code:`"edges"`
        ``"edges"`` builds the grid as the reference does, ``2 pi n_k / L_k`` along
        the Cartesian axes from the three edge lengths (cell angles ignored).
        ``"cell"`` builds it on the reciprocal lattice of the full cell,
        ``q = n B*`` with ``B* = 2 pi H^-T`` (``H`` the lower-triangular cell matrix),
        so that a tilted cell gets wavevectors whose phases do not change when a
        particle moves by a cell vector; ``dimensions`` may then have 6 entries
        (3 mean right angles), explicit ``wavevectors`` are Cartesian, and the cell
        is the one at construction time.  An orthorhombic cell gives the
        ``"edges"`` results.  No reference counterpart.
    parallel : `bool`, keyword-only
        Accepted for compatibility (the reference's numba thread switch).
    precision : `str`, keyword-only, default: :code:`"fp64"`
        ``"fp64"`` (default, ~1e-13 relative to the reference), or ``"fp32"``
        (lattice wavevectors only: phase factors and accumulation on the FP32
        pipe).  Each term carries ~1e-7 relative error, but the float32 sums run
        over chunks of up to 4,096 particles, so the worst-case error of rho(q) is
        ~1.5e-7 * N * min(N, 4096); on a 50,000-particle Lennard-Jones frame S(q)
        stays within 1e-3 relative, not 1e-6.
    kernel : `str`, keyword-only, optional
        GPU kernel strategy.  Default: chosen by the library -- for lattice
        wavevectors ``"lattice_dmma"`` (complex rank-N update on the FP64 matrix
        unit) from 16 (column group x nz tile) pairs up and ``"lattice_fp64"``
        (scalar DFMA) below, ``"general_fp64"`` (dot product + sincos) otherwise.

    Attributes
    ----------
    results.pairs, results.wavenumbers, results.ssf
        As in the reference.
    """

    def __init__(
            self, groups, groupings: Union[str, tuple] = "atoms", *,
            mode: str = None, form: str = "exp", dimensions=None,
            n_points: int = 32, n_surfaces: int = None,
            n_surface_points: int = 8, q_max: float = None,
            wavevectors: np.ndarray = None, sort: bool = True,
            unique: bool = True, parallel: bool = False, verbose: bool = True,
            precision: str = "fp64", kernel: str = None, host_com: bool = False,
            reciprocal: str = "edges", **kwargs) -> None:

        self._host_com = bool(host_com)
        self._groups = ([groups] if hasattr(groups, "universe")
                        and hasattr(groups, "positions") else list(groups))
        self.universe = self._groups[0].universe

        super().__init__(self.universe.trajectory, verbose, **kwargs)

        self._n_groups = len(self._groups)
        if isinstance(groupings, str):
            if groupings not in _GROUPINGS_SSF:
                emsg = (f"Invalid grouping '{groupings}'. Valid "
                        f"values: {', '.join(sorted(_GROUPINGS_SSF))}.")
                raise ValueError(emsg)
            self._groupings = self._n_groups * [groupings]
        else:
            if self._n_groups != len(groupings):
                emsg = ("The number of grouping values is not equal to "
                        "the number of groups.")
                raise ValueError(emsg)
            for g in groupings:
                if g not in _GROUPINGS_SSF:
                    emsg = (f"Invalid grouping '{g}'. Valid "
                            f"values: {', '.join(sorted(_GROUPINGS_SSF))}.")
                    raise ValueError(emsg)
            self._groupings = list(groupings)

        self._mode = mode
        if self._mode not in {None, "pair", "partial"}:
            raise ValueError("Invalid mode. Valid values: None, 'pair', "
                             "'partial'.")
        if self._mode == "pair" and not 1 <= len(self._groups) <= 2:
            emsg = "There must be exactly one or two groups when mode='pair'."
            raise ValueError(emsg)
        elif self._mode is None:
            if sum(g.n_atoms for g in self._groups) \
                    != self.universe.atoms.n_atoms:
                emsg = ("The provided atom groups do not contain all atoms "
                        "in the universe.")
                raise ValueError(emsg)
        if form not in {"exp", "trig"}:
            raise ValueError("Invalid form. Valid values: 'exp', 'trig'.")
        if precision not in {"fp64", "fp32"}:
            raise ValueError("Invalid precision. Valid values: 'fp64', 'fp32'.")

        if reciprocal not in {"edges", "cell"}:
            raise ValueError("Invalid reciprocal. Valid values: 'edges', 'cell'.")
        cell_mode = reciprocal == "cell"

        self._dimensions = None
        if dimensions is not None:
            if len(dimensions) != 3 and not (cell_mode and len(dimensions) == 6):
                raise ValueError("'dimensions' must have length 3"
                                 + (" or 6." if cell_mode else "."))
            self._dimensions = np.asarray(dimensions)
        elif self.universe.dimensions is not None:
            self._dimensions = self.universe.dimensions[
                :6 if cell_mode else 3].copy()
        elif wavevectors is None or cell_mode:
            raise ValueError("No system dimensions found or provided.")

        # reciprocal="cell": H of a tilted cell; the Fourier sums then run on
        # fractional coordinates s = r H^-1 (mdh_sq_set_cell) and take the
        # wavevectors as k = q H^T.  An orthorhombic cell keeps the "edges" path.
        self._cell = None
        if cell_mode:
            full = self._dimensions
            if len(full) == 3:
                full = np.concatenate((full, np.full(3, 90, full.dtype)))
            cell = _cell_matrices(full)[0]
            self._dimensions = full[:3]
            if not is_orthorhombic(full)[0]:
                self._cell = cell
                if n_surfaces:
                    raise ValueError("'n_surfaces' requires a cubic box.")

        # Wavevectors (reference: structure.py:1375-1416).  The grid spacing
        # uses the box edge as stored (float32 from the universe) promoted to
        # float64, and the np.meshgrid 'xy' ordering: row (i, j, k) of the
        # reshaped grid holds (g[j], g[i], g[k]).
        self._lattice_n = self._lattice_b = None
        if self._cell is not None:
            h = self._cell.astype(np.float64)
            if wavevectors is not None:
                self._wavevectors = np.asarray(wavevectors, dtype=np.float64)
                self._kvectors = self._wavevectors @ h.T
                self._lattice_n, self._lattice_b = _lattice_indices(
                    self._kvectors, np.ones(3))
            else:
                n = _grid_indices(n_points)
                self._wavevectors = n @ (2 * np.pi * np.linalg.inv(h).T)
                self._kvectors = 2 * np.pi * n
                self._lattice_n = n.astype(np.int32)
                self._lattice_b = np.full(3, 2 * np.pi)
        elif wavevectors is not None:
            self._wavevectors = np.asarray(wavevectors, dtype=np.float64)
            self._lattice_n, self._lattice_b = _lattice_indices(
                self._wavevectors, self._dimensions)
        else:
            cubic = np.allclose(self._dimensions, self._dimensions[0])
            idx = np.arange(n_points)
            if cubic:
                grids = 3 * [2 * np.pi * idx / self._dimensions[0]]
            else:
                grids = [2 * np.pi * idx / L for L in self._dimensions]
            n = _grid_indices(n_points)
            self._wavevectors = np.stack(
                (grids[0][n[:, 0]], grids[1][n[:, 1]], grids[2][n[:, 2]]), axis=-1
            )
            self._lattice_n = n.astype(np.int32)
            self._lattice_b = np.array([g[1] if n_points > 1 else 1.0
                                        for g in grids])
            if n_surfaces:
                if not cubic:
                    raise ValueError("'n_surfaces' requires a cubic box.")
                self._wavevectors = np.vstack(
                    (self._wavevectors,
                     _surface_wavevectors(grids[0], n_surfaces,
                                          n_surface_points))
                )
                self._lattice_n = self._lattice_b = None
        if self._cell is None:
            self._kvectors = self._wavevectors      # what sq_configure receives
        self._wavenumbers = np.linalg.norm(self._wavevectors, axis=1)

        if q_max is not None:
            keep = self._wavenumbers <= q_max
            self._wavevectors = self._wavevectors[keep]
            self._kvectors = self._kvectors[keep]
            self._wavenumbers = self._wavenumbers[keep]
            if self._lattice_n is not None:
                self._lattice_n = self._lattice_n[keep]

        self._Ns = np.fromiter(
            (_n_entities(a, g) for a, g in zip(self._groups, self._groupings)),
            dtype=int, count=self._n_groups
        )
        self._N = self._Ns.sum()
        self._form = form
        self._sort = sort
        self._unique = unique
        self._verbose = verbose
        self._precision = precision
        self._kernel = kernel

    def _prepare(self) -> None:
        # reference: structure.py:1456-1479
        self.results.pairs = (
            tuple(combinations_with_replacement(range(self._n_groups), 2))
            if self._mode == "partial"
            else ((0, self._n_groups - 1),) if self._mode == "pair"
            else ((None, None),)
        )
        self.results.ssf = np.zeros((len(self.results.pairs),
                                     len(self._wavenumbers)))
        self.results.wavenumbers = (np.unique(self._wavenumbers.round(11))
                                    if self._unique else self._wavenumbers)
        self.results.units = {"results.wavenumbers": "angstrom^-1"}

    def _begin(self, frames: np.ndarray):
        ctx = self._context()
        offsets = np.concatenate(([0], np.cumsum(self._Ns)))
        pairs = np.array([(-1, -1) if p[0] is None else p
                          for p in self.results.pairs], dtype=np.int32)
        if self._kernel is not None:
            mode = self._kernel
        elif self._lattice_n is None:
            mode = "general_fp64"
        else:
            mode = "lattice_fp32" if self._precision == "fp32" else "auto"
        ctx.sq_configure(int(self._N), offsets, self._kvectors, pairs,
                         lattice_n=self._lattice_n, lattice_b=self._lattice_b,
                         mode=mode)
        if self._cell is not None:
            ctx.sq_set_cell(self._cell)
        atoms_only = all(g == "atoms" for g in self._groupings)
        self._com = None
        if atoms_only:
            sets = [np.concatenate([g.ix for g in self._groups])]
            positions_fn = None
        else:
            plans = [_com_plan(g, gr) for g, gr in zip(self._groups, self._groupings)]
            if all(p is not None for p in plans) and len(plans) <= 8 \
                    and not getattr(self, "_host_com", False):
                # centres of mass on the device (com.cu), the groups written side by
                # side into one [frames, N, 3] buffer
                for slot, (starts, masses) in enumerate(plans):
                    ctx.com_configure(slot, starts, masses)
                self._com = [len(p[0]) - 1 for p in plans]
                return ([g.ix for g in self._groups], None,
                        12 * sum(g.n_atoms for g in self._groups))
            sets = [np.arange(self._N)]

            def positions_fn(ts):
                return [np.concatenate([
                    ts.positions[g.ix] if gr == "atoms"
                    else _centers_of_mass(g, gr, ts.positions[g.ix])
                    for g, gr in zip(self._groups, self._groupings)
                ])]
        return sets, positions_fn, 12 * int(self._N)

    def _staging_dtype(self, positions_fn):
        # centres of mass found on the host stay float64 up to the Fourier sums, as in
        # the reference's position buffer (structure.py:1468-1486)
        return np.float32 if positions_fn is None else np.float64

    def _consume(self, batch, device: bool = False) -> None:
        ptr, stride = batch.ptrs[0], batch.strides[0]
        f64 = batch.f64
        if self._com is not None:
            import torch
            N = int(self._N)
            # float64 centres of mass (the reference does not round them either)
            out = torch.empty((batch.n_frames, N, 3), dtype=torch.float64,
                              device=f"cuda:{self._device}")
            off = 0
            for slot, n in enumerate(self._com):
                self._ctx.com_reduce(slot, batch.ptrs[slot], batch.strides[slot],
                                     batch.n_frames, out.data_ptr() + 24 * off, 3 * N,
                                     device=device, f64=True)
                off += n
            ptr, stride, device, f64 = out.data_ptr(), 3 * N, True, True
        self._ctx.sq_accumulate(ptr, stride, batch.n_frames, device=device,
                                keepalive=batch.keepalive, f64=f64)
        _record(batch)

    def _finish(self) -> None:
        self._local_ssf = self._ctx.sq_fetch()

    def _conclude(self) -> None:
        # reference: structure.py:1529-1550
        self.results.ssf = all_reduce_sum(self._local_ssf, self._device)
        self.results.ssf /= self.n_frames * self._N

        if self._unique:
            # same columns, same order and same mean as the reference's
            # np.isclose(q, wavenumbers) loop; the memberships depend only on the
            # wavevectors, so they are found once per instance, not once per run
            if getattr(self, "_unique_members", None) is None:
                self._unique_members = _isclose_members(self.results.wavenumbers,
                                                        self._wavenumbers)
            self.results.ssf = _grouped_mean(self.results.ssf, self._unique_members)
        if self._sort:
            order = np.argsort(self.results.wavenumbers)
            self.results.wavenumbers = self.results.wavenumbers[order]
            self.results.ssf = self.results.ssf[:, order]


class IntermediateScatteringFunction(StructureFactor):
    r"""
    Coherent and incoherent (self) intermediate scattering functions
    :math:`F(q,\,t)`, :math:`F_\mathrm{s}(q,\,t)` and their partial variants,
    computed on the GPU (reference class: ``structure.py:1552-2127``).

    Same constructor as :class:`StructureFactor` plus

    dt : `float`, keyword-only, optional
        Time between frames (default: the trajectory's ``dt``).
    n_lags : `int`, keyword-only, optional
        Number of time lags (default: the number of analysed frames).
    incoherent : `bool`, keyword-only, default: :code:`False`
        Also compute the incoherent part (one direct sum per frame and lag over
        the particle displacements, as the reference does).

    Attributes
    ----------
    results.times, results.wavenumbers, results.pairs, results.cisf, results.iisf
        As in the reference: ``cisf`` has shape :math:`(N_t,\,N_\mathrm{pairs},
        \,N_q)`, ``iisf`` :math:`(N_t,\,N_\mathrm{groups},\,N_q)`.

    Notes
    -----
    * Time order matters, so under ``torch.distributed`` the *wavevectors* are
      sharded over the ranks (every rank streams all frames) and the columns are
      combined with one all-reduce.
    * ``rho(q, t)`` of every frame stays on the device (16 bytes per frame, group
      and wavevector), which is what the reference's comment at
      ``structure.py:1971-1977`` rules out for host memory; the incoherent part
      keeps a coordinate window of ``n_lags - 1`` frames.
    """

    def __init__(self, groups, groupings: Union[str, tuple] = "atoms", *,
                 mode: str = None, form: str = "exp", dimensions=None,
                 dt: float = None, n_points: int = 32, n_surfaces: int = None,
                 n_surface_points: int = 8, q_max: float = None,
                 wavevectors: np.ndarray = None, sort: bool = True,
                 unique: bool = True, n_lags: int = None,
                 incoherent: bool = False, parallel: bool = False,
                 verbose: bool = True, **kwargs) -> None:
        super().__init__(
            groups, groupings, mode=mode, form=form, dimensions=dimensions,
            n_points=n_points, n_surfaces=n_surfaces,
            n_surface_points=n_surface_points, q_max=q_max,
            wavevectors=wavevectors, sort=sort, unique=unique,
            parallel=parallel, verbose=verbose, **kwargs
        )
        self._dt = float(dt if dt is not None
                         else getattr(self._trajectory, "dt", 1.0))
        self._n_lags_arg = n_lags
        self._incoherent = incoherent

    def _prepare(self) -> None:
        # reference: structure.py:1899-1957
        self._n_lags = self._n_lags_arg or self.n_frames
        if self._n_lags > self.n_frames:
            raise ValueError("There are fewer frames than time lags.")
        df = 1
        if self.n_frames > 1:
            d = np.diff(self._frame_list)
            if d[0] <= 0 or not np.allclose(d, d[0]):
                emsg = ("The selected frames must be evenly spaced and "
                        "proceed forward in time.")
                raise ValueError(emsg)
            df = d[0]
        self.results.pairs = (
            tuple(combinations_with_replacement(range(self._n_groups), 2))
            if self._mode == "partial"
            else ((0, self._n_groups - 1),) if self._mode == "pair"
            else ((None, None),)
        )
        n_q = len(self._wavenumbers)
        self.results.cisf = np.zeros((
            self._n_lags,
            1 if self._mode is None else len(self.results.pairs), n_q))
        if self._incoherent:
            self.results.iisf = np.zeros((
                self._n_lags,
                1 if self._mode is None else self._n_groups, n_q))
        self.results.times = df * self._dt * np.arange(self._n_lags)
        self.results.wavenumbers = (np.unique(self._wavenumbers.round(11))
                                    if self._unique else self._wavenumbers)
        self.results.units = {"results.times": "picosecond",
                              "results.wavenumbers": "angstrom^-1"}

    def run(self, start: int = None, stop: int = None, step: int = None,
            frames=None, verbose: bool = None, **kwargs):
        """Performs the calculation (all ranks stream all frames; the wavevectors
        are sharded instead, see *Notes*)."""
        self._setup_frames(self._trajectory, start=start, stop=stop, step=step,
                           frames=frames)
        self._prepare()
        self.n_local_frames = self.n_frames
        self._process(self._frame_list)
        self._conclude()
        return self

    def _process(self, frames: np.ndarray) -> None:
        ctx = self._context()
        rank, size = world()
        n_q = len(self._wavenumbers)
        cols = np.array_split(np.arange(n_q), size)[rank]
        self._local_cols = cols
        offsets = np.concatenate(([0], np.cumsum(self._Ns)))
        pairs = np.array([(-1, -1) if p[0] is None else p
                          for p in self.results.pairs], dtype=np.int32)
        self._local = (np.zeros_like(self.results.cisf),
                       np.zeros_like(self.results.iisf)
                       if self._incoherent else None)
        if len(cols) == 0 or len(frames) == 0:
            return
        if self._kernel is not None:
            mode = self._kernel
        elif self._lattice_n is None:
            mode = "general_fp64"
        else:
            mode = "lattice_fp32" if self._precision == "fp32" else "auto"
        ctx.sq_configure(
            int(self._N), offsets, self._kvectors[cols], pairs,
            lattice_n=None if self._lattice_n is None else self._lattice_n[cols],
            lattice_b=self._lattice_b, mode=mode)
        if self._cell is not None:
            ctx.sq_set_cell(self._cell)
        ctx.isf_configure(self._n_lags, self._incoherent, len(frames))

        atoms_only = all(g == "atoms" for g in self._groupings)
        if atoms_only:
            sets = [np.concatenate([g.ix for g in self._groups])]
            positions_fn = None
        else:
            sets = [np.arange(self._N)]

            def positions_fn(ts):
                return [np.concatenate([
                    ts.positions[g.ix] if gr == "atoms"
                    else _centers_of_mass(g, gr, ts.positions[g.ix])
                    for g, gr in zip(self._groups, self._groupings)
                ])]

        # centres of mass stay float64 (reference: structure.py:1927-1957)
        feeder = FrameFeeder(self._trajectory, sets, frames,
                             self._default_batch(12 * int(self._N)),
                             positions_fn,
                             dtype=np.float32 if positions_fn is None else np.float64)
        for batch in feeder:
            ctx.isf_accumulate(batch.ptrs[0], batch.strides[0], batch.n_frames,
                               keepalive=batch.keepalive, f64=batch.f64)
            _record(batch)
        cisf, iisf = ctx.isf_fetch()
        self._local[0][:, :, cols] = cisf
        if self._incoherent:
            # the reference only fills the groups that form a (j, j) pair
            # (structure.py:2013-2027); with mode=None there is one row
            if self._mode is None:
                self._local[1][:, :, cols] = iisf
            else:
                for j in {j for j, k in self.results.pairs if j == k}:
                    self._local[1][:, j, cols] = iisf[:, j]

    def _conclude(self) -> None:
        # reference: structure.py:2087-2127
        self.results.cisf = all_reduce_sum(self._local[0], self._device)
        if self._incoherent:
            self.results.iisf = all_reduce_sum(self._local[1], self._device)
        normalization = (
            self._N * np.arange(self.n_frames,
                                self.n_frames - self._n_lags, -1)[:, None, None]
        )
        self.results.cisf = self.results.cisf / normalization
        if self._incoherent:
            self.results.iisf = self.results.iisf / normalization
        if self._unique:
            members = _isclose_members(self.results.wavenumbers, self._wavenumbers)
            self.results.cisf = _grouped_mean(self.results.cisf, members)
            if self._incoherent:
                self.results.iisf = _grouped_mean(self.results.iisf, members)
        if self._sort:
            order = np.argsort(self.results.wavenumbers)
            self.results.wavenumbers = self.results.wavenumbers[order]
            self.results.cisf = self.results.cisf[:, :, order]
            if self._incoherent:
                self.results.iisf = self.results.iisf[:, :, order]


def _isclose_members(unique_q: np.ndarray, wavenumbers: np.ndarray) -> list:
    """
    ``[np.flatnonzero(np.isclose(q, wavenumbers)) for q in unique_q]`` -- the groups
    the reference averages over in its ``_conclude`` methods (``structure.py:1538-1543``,
    ``polymer.py:1121-1128``) -- without the O(n_unique x n_q) scan: candidates come from
    a sorted copy (a window slightly wider than ``isclose``'s tolerance) and are then
    filtered with ``np.isclose`` itself, so the index sets are identical and ascending.
    """
    order = np.argsort(wavenumbers, kind="stable")
    w_sorted = wavenumbers[order]
    out = []
    for q in unique_q:
        tol = 1e-8 + 1.1e-5 * (abs(q) + 1e-8)          # isclose: atol + rtol * |w|
        lo = np.searchsorted(w_sorted, q - 2 * tol, side="left")
        hi = np.searchsorted(w_sorted, q + 2 * tol, side="right")
        cand = np.sort(order[lo:hi])
        out.append(cand[np.isclose(q, wavenumbers[cand])])
    return out


_GROUP_INDEX_CACHE = {}


def _grouped_mean(values: np.ndarray, members: list) -> np.ndarray:
    """
    ``np.stack([values[..., m].mean(axis=-1) for m in members], axis=-1)`` -- the
    reference's per-wavenumber averages (``structure.py:1538-1543``) -- with one numpy
    call per group SIZE instead of one per group: ``values[..., idx]`` with a 2-D index
    array ``[n_groups, size]`` keeps the memory layout of the per-group gather (index
    axes outermost), so the reduction over the last axis adds the same values in the
    same order (sequential for >= 2-D input, pairwise for 1-D) and the result is
    bit-identical to the loop (checked in ``tests/test_host.py``).
    """
    values = np.asarray(values)
    out = np.empty(values.shape[:-1] + (len(members),), dtype=np.float64)
    # the (groups, index array) pairs per group size depend on `members` only: built once per
    # membership list (the list object is kept by its analysis instance) and reused by every run
    plan = _GROUP_INDEX_CACHE.get(id(members))
    if plan is None or plan[0] is not members:
        by_size = {}
        for g, m in enumerate(members):
            by_size.setdefault(len(m), []).append(g)
        plan = (members, [(np.array(groups, dtype=np.intp),
                           np.array([members[g] for g in groups],
                                    dtype=np.intp).reshape(len(groups), size))
                          for size, groups in by_size.items()])
        if len(_GROUP_INDEX_CACHE) > 64:
            _GROUP_INDEX_CACHE.clear()
        _GROUP_INDEX_CACHE[id(members)] = plan
    for groups, idx in plan[1]:
        out[..., groups] = values[..., idx].mean(axis=-1)
    return out


def _closest_factor_pair(value: int) -> tuple:
    """
    Two factors of ``value`` that are close to each other, larger first: the
    greedy assignment of prime factors (largest first) to the slot that stays
    at or below ``round(sqrt(value))`` -- the same pairing as the reference's
    ``get_closest_factors(value, 2, reverse=True)``
    (``algorithm/utility.py:15-72``), which fixes how many polar and azimuthal
    points ``n_surface_points`` is split into.
    """
    root = float(value) ** 0.5
    root_int = int(np.round(root))
    if np.isclose(root, root_int):
        return root_int, root_int
    primes, rest, d = [], int(value), 2
    while d * d <= rest:
        while rest % d == 0:
            primes.append(d)
            rest //= d
        d += 1
    if rest > 1:
        primes.append(rest)
    slots, i = [1, 1], 0
    for j, f in enumerate(reversed(primes)):
        while i < 2:
            if slots[i] * f <= root_int or (j < 2 and slots[i] == 1):
                slots[i] *= f
                break
            i += 1
        else:
            slots[slots.index(min(slots))] *= f
    return max(slots), min(slots)


def _surface_wavevectors(grid: np.ndarray, n_surfaces: int,
                         n_surface_points: int) -> np.ndarray:
    """
    Extra off-lattice wavevectors on first-octant spherical surfaces of radii
    ``grid[1..n_surfaces]`` (reference: ``structure.py:1382-1403``).
    """
    n_theta, n_phi = _closest_factor_pair(n_surface_points)
    theta = np.linspace(np.pi / (2 * n_theta + 4),
                        np.pi / 2 - np.pi / (2 * n_theta + 4), n_theta)
    phi = np.linspace(np.pi / (2 * n_phi + 4),
                      np.pi / 2 - np.pi / (2 * n_phi + 4), n_phi)
    unit = np.stack((np.sin(theta) * np.cos(phi)[:, None],
                     np.sin(theta) * np.sin(phi)[:, None],
                     np.tile(np.cos(theta)[None, :], (n_phi, 1))), axis=-1)
    return np.einsum("o,tpd->otpd", grid[1:n_surfaces + 1], unit).reshape(
        (n_surfaces * n_surface_points, 3))
