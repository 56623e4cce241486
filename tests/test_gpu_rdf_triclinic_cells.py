"""GPU: the triclinic cell-list kernel (rdf_tri_cells_kernel) gives the counts of the
restated reference (the CPU oracle) and of the all-pairs triclinic kernel, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)              # rhombic dodecahedron
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)          # truncated octahedron
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)           # strongly tilted monoclinic


def _rp():
    from oracle import reference_port as rp
    return rp


def _S():
    from mdhelper_b200.analysis import structure
    return structure


def _widths(dims):
    h = _rp().triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    vol = abs(np.linalg.det(h))
    a, b, c = h
    return np.array([vol / np.linalg.norm(np.cross(b, c)), vol / np.linalg.norm(np.cross(c, a)),
                     vol / np.linalg.norm(np.cross(a, b))])


def _scaled(shape, L):
    return np.array([L * shape[0], L * shape[1], L * shape[2], *shape[3:]], np.float32)


def _universe(dims_list, n, seed, lo=0.0, hi=1.0):
    from mdhelper_b200.universe import SyntheticUniverse
    rng = np.random.default_rng(seed)
    dims = np.array(dims_list, np.float32)
    pos = np.empty((len(dims), n, 3), np.float32)
    for f, d in enumerate(dims):
        h = _rp().triclinic_vectors(d).astype(np.float64)
        pos[f] = ((rng.random((n, 3)) * (hi - lo) + lo) @ h).astype(np.float32)
    return SyntheticUniverse(pos, dims)


def _ctx_counts(p, cells, n_bins, rng_, mode, *, device=False, q=None, exclusion=None):
    """One accumulate call through the C ABI (same group unless q is given)."""
    import torch
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    F, n = p.shape[:2]
    ctx = _lib.Context(0)
    try:
        m = n if q is None else q.shape[1]
        ctx.rdf_configure(n, m, q is None, squared_thresholds(n_bins, rng_), rng_[0], rng_[1],
                          mode=mode, exclusion=exclusion)
        a, b = p, (p if q is None else q)
        if device:
            a = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            b = a if q is None else torch.from_numpy(np.ascontiguousarray(b)).cuda()
        ctx.rdf_accumulate_triclinic(a, 3 * n, b, 3 * m, cells, F, device=device)
        out = ctx.rdf_fetch()
        return out, ctx.rdf_pair_evaluations()
    finally:
        ctx.close()


def _cells_of(dims):
    return np.stack([_rp().triclinic_vectors(d) for d in np.atleast_2d(dims)]).astype(np.float32)


ORACLE_CELLS = [(10.5, 11.25, 12.0, 75.0, 82.0, 64.0), (10.0, 11.5, 12.5, 90.0, 90.0, 70.0),
                (11.0, 11.0, 11.0, 60.0, 60.0, 60.0), _scaled(RD, 12.0), _scaled(TO, 12.0),
                _scaled(TILT, 12.0)]


@pytest.mark.parametrize("dims", ORACLE_CELLS, ids=range(len(ORACLE_CELLS)))
def test_cells_mode_matches_the_oracle(dims):
    """Same group, two groups of unequal size, exclusions (3, 3) and (2, 5), r_lo > 0,
    1, 70 and 1000 bins, coordinates up to 2 cells outside the box, two frames."""
    u = _universe([dims, dims], 2400, seed=int(sum(dims)), lo=-2.0, hi=3.0)
    r_hi = float(_widths(dims).min() / 3.3)
    a, b = u.select(slice(0, 900)), u.select(slice(900, 2400))
    S = _S()
    cases = [((u.atoms, None), None, 70, (0.0, r_hi)),
             ((a, b), None, 1000, (0.0, r_hi)),
             ((u.atoms, None), (3, 3), 1, (0.0, r_hi)),
             ((a, b), (2, 5), 70, (0.4 * r_hi, r_hi)),
             ((u.atoms, None), None, 1000, (0.3 * r_hi, r_hi))]
    for (g1, g2), excl, n_bins, rng_ in cases:
        kw = dict(n_bins=n_bins, range=rng_, exclusion=excl)
        want = _rp().rdf_run(u, g1, g2, **kw)
        r = S.RadialDistributionFunction(g1, g2, verbose=False, mode="cells", **kw).run()
        assert np.array_equal(r.results.counts, want["counts"]), (excl, n_bins, rng_)
        np.testing.assert_allclose(r.results.rdf, want["rdf"], rtol=1e-6)


def test_exactly_three_cells_on_one_axis():
    from mdhelper_b200 import _lib
    dims = _scaled(TO, 12.0)
    r_hi = float(_widths(dims).min() / 3.2)
    nc, _ = _lib.triclinic_grid(_cells_of(dims)[0], r_hi, 3000)
    assert min(nc) == 3
    u = _universe([dims], 3000, seed=3)
    p = u.trajectory.coordinates[0]
    got = _S().radial_histogram(p, p, 50, (0.0, r_hi), dims, mode="cells")
    assert np.array_equal(got, _rp().radial_histogram(p, p, 50, (0.0, r_hi), dims))


def _lattice_pairs(dims, r_hi, edges, rng):
    """Particles near the corners, edges and faces of the cell and partners at distances
    at or next to r_hi and the bin edges, in directions whose nearest image crosses one,
    two or three periodic faces (every sign pattern of m')."""
    h = _rp().triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    one_m = np.nextafter(1.0, 0.0)
    spots = [0.0, 1e-6, 0.01, 0.5, 0.99, one_m]
    lengths = np.concatenate([[r_hi * (1 - 1e-7), r_hi, r_hi * (1 + 1e-7)],
                              edges[1:-1], edges[1:-1] * (1 + 1e-7), edges[1:-1] * (1 - 1e-7)])
    first, second = [], []
    for fa in spots:
        for fb in spots:
            for fc in spots:
                fr = np.array([fa, fb, fc])
                base = fr @ h
                for _ in range(3):
                    # outward where the particle is near a face: the partner wraps
                    sgn = np.where(fr > 0.5, 1.0, np.where(fr < 0.5, -1.0, rng.choice([-1, 1], 3)))
                    v = np.abs(rng.normal(size=3)) * sgn
                    v /= np.linalg.norm(v)
                    first.append(base)
                    second.append(base + v * rng.choice(lengths))
    return np.concatenate([first, second]).astype(np.float32)


@pytest.mark.parametrize("shape", [RD, TO, TILT])
@pytest.mark.parametrize("scale,cells", [(9.0, 3.05), (20.0, 5.5)])
def test_adversarial_lattice(shape, scale, cells):
    dims = _scaled(shape, scale)
    r_hi = float(_widths(dims).min() / cells)
    edges = np.linspace(0.0, r_hi, 41)
    p = _lattice_pairs(dims, r_hi, edges, np.random.default_rng(5))
    want = _rp().radial_histogram(p, p, 40, (0.0, r_hi), dims)
    got = _S().radial_histogram(p, p, 40, (0.0, r_hi), dims, mode="cells")
    assert want.sum() > 0
    assert np.array_equal(got, want)
    q = p[::-1].copy()                                # two groups: the full stencil
    want = _rp().radial_histogram(p, q, 40, (0.2 * r_hi, r_hi), dims)
    got = _S().radial_histogram(p, q, 40, (0.2 * r_hi, r_hi), dims, mode="cells")
    assert np.array_equal(got, want)


def _fluid(n, dims, rng, cluster=0.0):
    h = _rp().triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    p = (rng.random((n, 3)) * 1.2 - 0.1) @ h
    k = int(cluster * n)
    if k:
        p[:k] = p[0] + rng.normal(scale=0.6, size=(k, 3))
    return p.astype(np.float32)


def test_at_scale_equals_the_all_pairs_kernel():
    """80k particles: a multi-frame call with a different cell in every frame (triclinic
    NPT), a dense cluster, NaN coordinates in one frame, host and device input, one group
    and two groups."""
    rng = np.random.default_rng(11)
    n, F = 80000, 3
    L = (n / 0.8) ** (1 / 3)
    shapes = [RD, TO, TILT]
    dims = np.stack([_scaled(s, L * (1 + 0.01 * f)) for f, s in enumerate(shapes)])
    p = np.stack([_fluid(n, dims[f], rng, cluster=0.15 if f == 1 else 0.0) for f in range(F)])
    p[2, 17] = np.nan
    p[2, 4000, 1] = np.nan
    cells = _cells_of(dims)
    for kw in [dict(), dict(device=True), dict(exclusion=(4, 4))]:
        want, ev_all = _ctx_counts(p, cells, 100, (0.0, 2.5), "allpairs", **kw)
        got, ev = _ctx_counts(p, cells, 100, (0.0, 2.5), "cells", **kw)
        assert want.sum() > 0
        assert np.array_equal(got, want), kw
        assert ev < ev_all / 50
    q = p[:, :30000].copy()
    want, _ = _ctx_counts(p[:, 30000:].copy(), cells, 64, (0.5, 2.5), "allpairs", q=q)
    got, _ = _ctx_counts(p[:, 30000:].copy(), cells, 64, (0.5, 2.5), "cells", q=q)
    assert np.array_equal(got, want)


def test_coordinates_far_outside_the_cell():
    """A frame with a coordinate a long way out of the cell (beyond what the margin
    covers) is counted with the 27-image arithmetic for every pair: same counts."""
    rng = np.random.default_rng(2)
    dims = _scaled(TO, 20.0)
    p = _fluid(6000, dims, rng)[None].repeat(2, 0)
    p[1, 5] = [1.0e20, -3.0e19, 5.0e19]     # the wrap cannot bring it back exactly
    cells = _cells_of(np.stack([dims, dims]))
    want, _ = _ctx_counts(p, cells, 30, (0.0, 3.0), "allpairs")
    got, _ = _ctx_counts(p, cells, 30, (0.0, 3.0), "cells")
    assert np.array_equal(got, want)


def test_class_auto_picks_the_cell_list_and_mixes_cell_kinds():
    from mdhelper_b200.universe import SyntheticUniverse
    rng = np.random.default_rng(8)
    n = 4000
    L = (n / 0.8) ** (1 / 3)
    tri = _scaled(RD, L * 1.2)
    ortho = np.array([L, L, L, 90, 90, 90], np.float32)
    dims = np.stack([tri, ortho, _scaled(TO, L * 1.2)])
    pos = np.stack([_fluid(n, d, rng) for d in dims])
    u = SyntheticUniverse(pos, dims)
    S = _S()
    kw = dict(n_bins=60, range=(0.0, 2.5), verbose=False)
    auto = S.RadialDistributionFunction(u.atoms, **kw).run()
    full = S.RadialDistributionFunction(u.atoms, mode="allpairs", **kw).run()
    assert np.array_equal(auto.results.counts, full.results.counts)
    np.testing.assert_allclose(auto.results.rdf, full.results.rdf, rtol=1e-12)
    assert auto._pair_evaluations < 0.25 * n * n * 3
    want = _rp().rdf_run(u, u.atoms, n_bins=60, range=(0.0, 2.5))
    assert np.array_equal(auto.results.counts, want["counts"])
    # triclinic frames alone: auto takes the cell list there too
    ut = SyntheticUniverse(pos[[0, 2]].copy(), dims[[0, 2]].copy())
    a = S.RadialDistributionFunction(ut.atoms, **kw).run()
    assert a._pair_evaluations < 0.25 * n * n * 2


def test_too_few_cells_raise():
    dims = _scaled(RD, 10.0)
    u = _universe([dims], 500, seed=1)
    r_hi = float(_widths(dims).min() / 2.9)
    with pytest.raises(ValueError, match="cell-list mode"):
        _S().RadialDistributionFunction(u.atoms, n_bins=10, range=(0.0, r_hi), verbose=False,
                                        mode="cells").run()
