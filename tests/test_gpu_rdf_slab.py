"""GPU: two-dimensional RDFs (drop_axis) on the cell lists -- one cell along the dropped
axis, the 9-cell stencil of the plane -- and on triclinic cells.  Counts are compared with
np.array_equal against the all-pairs kernels and the restated reference (the CPU oracle)."""
import numpy as np
import pytest

from conftest import universe_from
from test_gpu_rdf import VARIANTS
from test_oracle import rdf_groups, rdf_kwargs

pytestmark = pytest.mark.gpu


def _rp():
    from oracle import reference_port as rp
    return rp


def _S():
    from mdhelper_b200.analysis import structure
    return structure


def _U(pos, dims):
    from mdhelper_b200.universe import SyntheticUniverse
    return SyntheticUniverse(np.asarray(pos, np.float32), np.asarray(dims, np.float32))


def _rdf(g1, g2=None, **kw):
    return _S().RadialDistributionFunction(g1, g2, verbose=False, **kw).run()


# ---- the stored reference outputs -------------------------------------------------------------

@pytest.mark.parametrize("hist,arith", VARIANTS + [("warp_atomic", "audit")])
@pytest.mark.parametrize("name", ["dropz", "dropx_density"])
def test_golden_drop_axis_cases_on_the_cell_list(golden, name, hist, arith):
    """The stored cases' 9.09 box holds 2 cells of their range (0, 3.5): the range is
    shortened to fit 3, and the oracle gives the counts there."""
    g = golden(f"rdf_{name}")
    u = universe_from(g)
    ag1, ag2 = rdf_groups(u, g)
    kw = rdf_kwargs(g)
    if name == "dropx_density":
        kw["norm"] = "density"
    lmin = float(np.atleast_2d(g["dims"])[:, :3].min())
    kw["range"] = (kw["range"][0], np.float32(lmin / 3.2).item())
    want = _rp().rdf_run(u, ag1, ag2, **kw)
    assert want["counts"].sum() > 0
    r = _rdf(ag1, ag2, mode="cells", hist=hist, arith=arith, **kw)
    assert np.array_equal(r.results.counts, want["counts"])
    np.testing.assert_allclose(r.results.rdf, want["rdf"], rtol=1e-6)
    full = _rdf(ag1, ag2, mode="allpairs", hist=hist, arith=arith, **kw)
    assert np.array_equal(full.results.counts, want["counts"])
    if arith in ("auto", "audit"):
        assert r._filter_stats["eligible"] == 1
        assert r._filter_stats["audit_violations"] == 0


# ---- orthorhombic slabs -------------------------------------------------------------------

def _slab(n, drop, edges, rng, thick=2.0, lo=0.0, hi=1.0):
    """n particles of a layer normal to the dropped axis: uniform over the kept edges
    (fractions lo .. hi of them), a thin spread along the dropped one (zeroed anyway)."""
    p = np.empty((n, 3))
    for k in range(3):
        if k == drop:
            p[:, k] = 0.5 * edges[k] + thick * (rng.random(n) - 0.5)
        else:
            p[:, k] = (lo + (hi - lo) * rng.random(n)) * edges[k]
    return p.astype(np.float32)


def _edges(n, drop, rho2=0.8, aspect=1.1):
    L = np.sqrt(n / rho2 / aspect)
    e = np.array([L, L * aspect, 0.0])
    e = np.insert(e[:2], drop, 30.0)
    return e.astype(np.float32)


def _three_ways(u, g1, g2=None, oracle=True, **kw):
    """cells == all-pairs (== oracle); returns the cell-list run."""
    kw.setdefault("norm", None)
    wrap = kw.pop("wrap", "auto")
    arith = kw.pop("arith", "auto")
    cells = _rdf(g1, g2, mode="cells", wrap=wrap, arith=arith, **kw)
    full = _rdf(g1, g2, mode="allpairs", wrap=wrap, arith=arith, **kw)
    assert cells.results.counts.sum() > 0
    assert np.array_equal(cells.results.counts, full.results.counts), kw
    if oracle:
        method = {"auto": None, "never": "bruteforce", "always": "nsgrid"}[wrap]
        want = _rp().rdf_run(u, g1, g2, method=method, **kw)
        assert np.array_equal(cells.results.counts, want["counts"]), kw
    n1 = g1.n_atoms
    assert cells._pair_evaluations < 0.02 * n1 * (n1 if g2 is None else g2.n_atoms) * \
        len(u.trajectory)
    return cells


@pytest.mark.parametrize("drop", [0, 1, 2])
def test_orthorhombic_slabs(drop):
    """50k particles: same group and two groups, exclusions (1, 1) and (2, 5), r_lo > 0
    with 1000 bins, the fp32 filter audited and the fp64 kernel alone."""
    rng = np.random.default_rng(100 + drop)
    n = 50_000
    e = _edges(n, drop)
    dims = np.array([*e, 90, 90, 90], np.float32)
    u = _U(_slab(n, drop, e, rng)[None], dims)
    a, b = u.select(slice(0, 30_000)), u.select(slice(30_000, n))
    r = _three_ways(u, u.atoms, n_bins=100, range=(0.0, 2.5), drop_axis=drop)
    assert r._filter_stats["eligible"] == 1
    _three_ways(u, a, b, n_bins=100, range=(0.0, 2.5), drop_axis=drop)
    _three_ways(u, u.atoms, n_bins=50, range=(0.0, 3.0), drop_axis=drop, exclusion=(1, 1))
    _three_ways(u, a, b, n_bins=1000, range=(0.7, 2.5), drop_axis=drop, exclusion=(2, 5))
    _three_ways(u, u.atoms, n_bins=1000, range=(0.5, 2.0), drop_axis=drop, arith="off")
    for g1, g2 in [(u.atoms, None), (a, b)]:
        st = _rdf(g1, g2, mode="cells", arith="audit", n_bins=80, range=(0.0, 2.5),
                  drop_axis=drop, norm=None)._filter_stats
        assert st["eligible"] == 1 and st["audit_violations"] == 0, st


@pytest.mark.parametrize("drop", [0, 1, 2])
def test_orthorhombic_slabs_outside_the_box_and_changing_boxes(drop):
    """Coordinates up to a box outside the cell under wrap auto / never / always; a box
    that changes from frame to frame (also along the dropped axis: the widened edge)."""
    rng = np.random.default_rng(200 + drop)
    n, F = 50_000, 3
    e = _edges(n, drop)
    dims = np.stack([np.array([*(e * (1 + 0.03 * f)), 90, 90, 90], np.float32)
                     for f in range(F)])
    pos = np.stack([_slab(n, drop, dims[f, :3], rng, lo=-1.0, hi=2.0) for f in range(F)])
    u = _U(pos, dims)
    for wrap in ("auto", "never", "always"):
        # the oracle's brute force (wrap="never") is too slow for 50k particles on the CPU:
        # it checks a 6k-particle group of the same frames instead
        _three_ways(u, u.atoms, n_bins=60, range=(0.0, 2.5), drop_axis=drop, wrap=wrap,
                    oracle=wrap != "never")
    small = u.select(slice(0, 6_000))
    _three_ways(u, small, n_bins=60, range=(0.0, 2.5), drop_axis=drop, wrap="never")
    a, b = u.select(slice(0, 20_000)), u.select(slice(20_000, n))
    _three_ways(u, a, b, n_bins=60, range=(0.3, 2.5), drop_axis=drop, wrap="always")


@pytest.mark.parametrize("drop", [0, 2])
def test_orthorhombic_slab_with_a_dense_cluster(drop):
    """A cluster far denser than the layer: cells with more particles than one warp's
    buffer go to the fp64 kernel (crowded-cell path), longer candidate lists are done in
    segments."""
    rng = np.random.default_rng(300 + drop)
    n = 50_000
    e = _edges(n, drop)
    dims = np.array([*e, 90, 90, 90], np.float32)
    p = _slab(n, drop, e, rng).astype(np.float64)
    kept = [k for k in range(3) if k != drop]
    centre = 0.5 * e.astype(np.float64)
    p[:4000, kept] = centre[kept] + 0.35 * rng.standard_normal((4000, 2))
    p[4000:5500, kept] = (np.array([0.02, 0.98]) * e[kept]
                          + 0.8 * rng.standard_normal((1500, 2)))   # across a face
    u = _U(p.astype(np.float32)[None], dims)
    a, b = u.select(slice(0, 30_000)), u.select(slice(30_000, n))
    for arith in ("auto", "audit", "off"):
        _three_ways(u, u.atoms, n_bins=90, range=(0.0, 3.0), drop_axis=drop, arith=arith)
    _three_ways(u, a, b, n_bins=90, range=(0.0, 3.0), drop_axis=drop, exclusion=(4, 4))


# ---- triclinic cells ----------------------------------------------------------------------------

HEX120 = (1.0, 1.0, 0.8, 90.0, 90.0, 120.0)
HEX60 = (1.0, 1.0, 0.8, 90.0, 90.0, 60.0)
TILTED_C = (1.0, 1.1, 0.9, 72.0, 112.0, 90.0)


def _tri_universe(shapes, L, n, seed, lo=0.0, hi=1.0, drop=2):
    """Particles uniform in fractional coordinates lo .. hi of each cell (the dropped axis
    is zeroed by the analysis anyway)."""
    rng = np.random.default_rng(seed)
    dims = np.array([[L * s[0], L * s[1], L * s[2], *s[3:]] for s in shapes], np.float32)
    pos = np.empty((len(dims), n, 3), np.float32)
    for f, d in enumerate(dims):
        h = _rp().triclinic_vectors(d).astype(np.float64)
        pos[f] = ((rng.random((n, 3)) * (hi - lo) + lo) @ h).astype(np.float32)
    return _U(pos, dims)


def _plane_min_width(dims):
    d = np.asarray(dims, np.float32).copy()
    d[2] = d[:3].max()
    h = _rp().triclinic_vectors(d).astype(np.float64)
    return min(h[0, 0] * h[1, 1] / np.hypot(h[1, 0], h[1, 1]), h[1, 1])


@pytest.mark.parametrize("shape", [HEX120, HEX60, TILTED_C], ids=["hex120", "hex60", "tilted_c"])
def test_triclinic_drop_z_cell_list(shape):
    """drop_axis=2: same group and two groups, exclusions, r_lo > 0, 1000 bins, coordinates
    outside the cell, two frames; results.rdf within 1e-6 of the reference's."""
    u = _tri_universe([shape, shape], 60.0, 2000, seed=int(shape[3] + shape[5]), lo=-1.0, hi=2.0)
    r_hi = float(_plane_min_width([60.0 * x for x in shape[:3]] + list(shape[3:])) / 5.3)
    a, b = u.select(slice(0, 800)), u.select(slice(800, 2000))
    cases = [((u.atoms, None), None, 70, (0.0, r_hi)),
             ((a, b), None, 1000, (0.0, r_hi)),
             ((u.atoms, None), (2, 2), 40, (0.0, r_hi)),
             ((a, b), (2, 5), 70, (0.4 * r_hi, r_hi))]
    for (g1, g2), excl, n_bins, rng_ in cases:
        kw = dict(n_bins=n_bins, range=rng_, exclusion=excl, drop_axis=2)
        want = _rp().rdf_run(u, g1, g2, **kw)
        assert want["counts"].sum() > 0
        cells = _rdf(g1, g2, mode="cells", **kw)
        full = _rdf(g1, g2, mode="allpairs", **kw)
        assert np.array_equal(cells.results.counts, want["counts"]), (excl, n_bins, rng_)
        assert np.array_equal(full.results.counts, want["counts"]), (excl, n_bins, rng_)
        np.testing.assert_allclose(cells.results.rdf, want["rdf"], rtol=1e-6)
        assert cells._pair_evaluations < 0.5 * full._pair_evaluations


@pytest.mark.parametrize("drop", [0, 1])
@pytest.mark.parametrize("shape", [HEX120, TILTED_C], ids=["hex120", "tilted_c"])
def test_triclinic_drop_x_or_y_runs_all_pairs(shape, drop):
    """drop_axis 0 or 1 on a triclinic cell: the wrap moves the zeroed coordinate again (a
    tilted cell), which the 27-image kernel follows; the cell list refuses it and auto
    takes all pairs."""
    u = _tri_universe([shape, shape], 14.0, 1500, seed=drop + 7, lo=-0.5, hi=1.5)
    for excl, rng_ in [(None, (0.0, 4.0)), ((3, 3), (1.0, 6.0))]:
        kw = dict(n_bins=50, range=rng_, exclusion=excl, drop_axis=drop)
        want = _rp().rdf_run(u, u.atoms, **kw)
        assert want["counts"].sum() > 0
        for mode in ("allpairs", "auto"):
            r = _rdf(u.atoms, mode=mode, **kw)
            assert np.array_equal(r.results.counts, want["counts"]), (mode, excl)
            np.testing.assert_allclose(r.results.rdf, want["rdf"], rtol=1e-6)
    with pytest.raises(ValueError, match="drop_axis 2"):
        _rdf(u.atoms, mode="cells", n_bins=10, range=(0.0, 2.0), drop_axis=drop)


def test_triclinic_drop_z_at_scale_equals_all_pairs():
    """60k particles in a hexagonal layer, three frames with changing cells, a dense
    cluster, host and device input, one and two groups."""
    import torch
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    rng = np.random.default_rng(17)
    n, F = 60_000, 3
    L = np.sqrt(n / 0.8 / np.sin(np.pi / 3))
    dims = np.stack([np.array([L * (1 + 0.01 * f), L, L, 90, 90, 120 - 5 * f], np.float32)
                     for f in range(F)])
    cells = np.stack([_rp().triclinic_vectors(d) for d in dims]).astype(np.float32)
    p = np.empty((F, n, 3), np.float32)
    for f in range(F):
        q = rng.random((n, 3)) @ cells[f].astype(np.float64)
        q[:2000, :2] = q[0, :2] + 0.5 * rng.standard_normal((2000, 2))
        q[:, 2] = 0.0
        p[f] = q
    for kw in [dict(), dict(device=True), dict(exclusion=(4, 4))]:
        out = {}
        for mode in ("allpairs", "cells"):
            ctx = _lib.Context(0)
            try:
                ctx.rdf_configure(n, n, True, squared_thresholds(100, (0.0, 2.5)), 0.0, 2.5,
                                  mode=mode, drop_axis=2, exclusion=kw.get("exclusion"))
                a = torch.from_numpy(p).cuda() if kw.get("device") else p
                ctx.rdf_accumulate_triclinic(a, 3 * n, a, 3 * n, cells, F,
                                             device=bool(kw.get("device")))
                out[mode] = (ctx.rdf_fetch(), ctx.rdf_pair_evaluations())
            finally:
                ctx.close()
        assert out["cells"][0].sum() > 0
        assert np.array_equal(out["cells"][0], out["allpairs"][0]), kw
        assert out["cells"][1] < out["allpairs"][1] / 50


# ---- kernel choice, mixed trajectories, errors -----------------------------------------------

def test_auto_picks_the_cell_list_for_large_slabs_only():
    rng = np.random.default_rng(5)
    n = 40_000
    e = _edges(n, 2)
    dims = np.array([*e, 90, 90, 90], np.float32)
    u = _U(_slab(n, 2, e, rng)[None], dims)
    kw = dict(n_bins=50, range=(0.0, 2.5), drop_axis=2, norm=None)
    auto = _rdf(u.atoms, **kw)
    assert auto._pair_evaluations < 0.01 * n * n
    want = _rp().rdf_run(u, u.atoms, **kw)
    assert np.array_equal(auto.results.counts, want["counts"])
    # small: all pairs
    small = u.select(slice(0, 1500))
    assert _rdf(small, **kw)._pair_evaluations >= 1500 * 1500 / 2
    # a kept edge shorter than 4 cut-offs: all pairs (the dropped one does not count)
    thin = np.array([e[0], 9.0, 30.0, 90, 90, 90], np.float32)
    ut = _U(_slab(n, 1, thin[:3], rng)[None], thin)
    assert _rdf(ut.atoms, **kw)._pair_evaluations >= n * n / 2
    ut1 = _rdf(ut.atoms, **{**kw, "drop_axis": 1})
    assert ut1._pair_evaluations < 0.01 * n * n
    # triclinic drop z: the flat cell list (the all-pairs kernel gives the counts here: the
    # oracle's 27-image brute force is too slow for 40k particles)
    L = float(np.sqrt(n / 0.8 / np.sin(np.pi / 3)))
    hexd = np.array([L, L, 20.0, 90, 90, 120], np.float32)
    h = _rp().triclinic_vectors(np.array([L, L, L, 90, 90, 120], np.float32)).astype(np.float64)
    ph = (rng.random((n, 3)) @ h).astype(np.float32)
    uh = _U(ph[None], hexd)
    a = _rdf(uh.atoms, **kw)
    assert a._pair_evaluations < 0.01 * n * n
    full = _rdf(uh.atoms, mode="allpairs", **kw)
    assert np.array_equal(a.results.counts, full.results.counts)
    # c almost in the plane: after widening to |c| = L, c_z = L sin(0.5 deg) < r_max + M,
    # so auto takes all pairs and mode="cells" refuses
    steep = np.array([L, L, 20.0, 90.0, 0.5, 90.0], np.float32)
    hs = _rp().triclinic_vectors(np.array([L, L, L, 90.0, 0.5, 90.0], np.float32))
    assert 0 < hs[2, 2] < 2.5
    us = _U(ph[None], steep)
    assert _rdf(us.atoms, **kw)._pair_evaluations >= n * n
    with pytest.raises(ValueError, match="c_z"):
        _rdf(us.atoms, mode="cells", **kw)


def test_mixed_orthorhombic_and_triclinic_trajectory_with_drop_axis():
    rng = np.random.default_rng(9)
    n = 3000
    L = 60.0
    dims = np.array([[L, L * 1.05, 40.0, 90, 90, 120], [L, L, 40.0, 90, 90, 90],
                     [L * 1.02, L, 40.0, 90, 90, 60]], np.float32)
    pos = np.stack([(rng.random((n, 3)) * [L, L, 40.0]).astype(np.float32) for _ in dims])
    u = _U(pos, dims)
    kw = dict(n_bins=60, range=(0.0, 9.0), drop_axis=2)
    want = _rp().rdf_run(u, u.atoms, **kw)
    for mode in ("auto", "allpairs", "cells"):
        r = _rdf(u.atoms, mode=mode, **kw)
        assert np.array_equal(r.results.counts, want["counts"]), mode
        np.testing.assert_allclose(r.results.rdf, want["rdf"], rtol=1e-6)
        np.testing.assert_allclose(r._area_or_volume, want["volume"], rtol=1e-6)
    kw["drop_axis"] = 0
    want = _rp().rdf_run(u, u.atoms, **kw)
    r = _rdf(u.atoms, **kw)
    assert np.array_equal(r.results.counts, want["counts"])
    np.testing.assert_allclose(r.results.rdf, want["rdf"], rtol=1e-6)


def test_cell_list_errors_with_drop_axis():
    rng = np.random.default_rng(4)
    # a kept edge shorter than 3 cut-offs; the dropped edge may be as short as it likes
    dims = np.array([30.0, 2.0, 7.0, 90, 90, 90], np.float32)
    u = _U((rng.random((1, 2000, 3)) * dims[:3]).astype(np.float32), dims)
    with pytest.raises(ValueError, match="cell-list mode"):
        _rdf(u.atoms, mode="cells", n_bins=10, range=(0.0, 2.5), drop_axis=2)
    r = _rdf(u.atoms, mode="cells", n_bins=10, range=(0.0, 2.3), drop_axis=1, norm=None)
    want = _rp().rdf_run(u, u.atoms, n_bins=10, range=(0.0, 2.3), drop_axis=1, norm=None)
    assert np.array_equal(r.results.counts, want["counts"])
