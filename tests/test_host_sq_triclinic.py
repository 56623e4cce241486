"""CPU: wavevectors on the reciprocal lattice of a triclinic cell (StructureFactor
reciprocal="cell") and the fp64 map of coordinates to fractional coordinates that
mdh_sq_set_cell applies before the Fourier sums (common.cuh tri_frac)."""
import numpy as np
import pytest

from mdhelper_b200 import _lib
from mdhelper_b200.analysis import structure as S
from mdhelper_b200.analysis._triclinic import triclinic_vectors
from mdhelper_b200.universe import SyntheticUniverse

CELLS = {
    "monoclinic": (9.0, 10.0, 11.0, 90.0, 104.0, 90.0),
    "hexagonal": (9.0, 9.0, 12.0, 90.0, 90.0, 120.0),
    "rhombic_dodecahedron": (10.0, 10.0, 10.0, 60.0, 60.0, 90.0),
    "truncated_octahedron": (10.0, 10.0, 10.0, 70.53, 109.47, 70.53),
}
LD = np.longdouble
U = 2.0 ** -53


def _universe(dims, n=40, seed=0):
    rng = np.random.default_rng(seed)
    h = triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    pos = (rng.random((1, n, 3)) @ h).astype(np.float32)
    return SyntheticUniverse(pos, np.asarray(dims, np.float32))


def _xy_indices(n_points):
    idx = np.arange(n_points)
    return np.stack(np.meshgrid(idx, idx, idx), -1).reshape(-1, 3)


@pytest.mark.parametrize("dims", [(9.0, 10.0, 11.0), (9.0, 10.0, 11.0, 90.0, 90.0, 90.0),
                                  (10.0, 10.0, 10.0, 90.0, 90.0, 90.0)])
@pytest.mark.parametrize("q_max", [None, 2.1])
def test_orthorhombic_cell_grid_is_the_edges_grid(dims, q_max):
    u = _universe((*dims[:3], 90.0, 90.0, 90.0))
    e = S.StructureFactor(u.atoms, n_points=7, q_max=q_max, verbose=False)
    c = S.StructureFactor(u.atoms, n_points=7, q_max=q_max, verbose=False,
                          reciprocal="cell")
    cd = S.StructureFactor(u.atoms, n_points=7, q_max=q_max, verbose=False,
                           reciprocal="cell", dimensions=np.asarray(dims, np.float32))
    for s in (c, cd):
        assert s._cell is None
        for name in ("_wavevectors", "_kvectors", "_wavenumbers", "_lattice_n", "_lattice_b"):
            assert np.array_equal(getattr(s, name), getattr(e, name)), name


@pytest.mark.parametrize("name", sorted(CELLS))
@pytest.mark.parametrize("q_max", [None, 1.7])
def test_triclinic_grid_is_n_times_the_reciprocal_basis(name, q_max):
    dims = CELLS[name]
    u = _universe(dims)
    s = S.StructureFactor(u.atoms, n_points=6, q_max=q_max, verbose=False,
                          reciprocal="cell")
    h = triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    assert np.array_equal(s._cell, triclinic_vectors(np.asarray(dims, np.float32)))
    bstar = 2 * np.pi * np.linalg.inv(h).T
    np.testing.assert_allclose(bstar @ h.T, 2 * np.pi * np.eye(3), atol=1e-13)
    n = _xy_indices(6)
    q = n @ bstar
    keep = np.ones(len(n), bool) if q_max is None else np.linalg.norm(q, axis=1) <= q_max
    assert keep.sum() < len(n) or q_max is None
    np.testing.assert_allclose(s._wavevectors, q[keep], rtol=1e-15, atol=1e-15)
    assert np.array_equal(s._lattice_n, n[keep])
    assert np.array_equal(s._kvectors, 2 * np.pi * n[keep])
    assert np.array_equal(s._lattice_b, np.full(3, 2 * np.pi))
    assert np.array_equal(s._wavenumbers, np.linalg.norm(s._wavevectors, axis=1))
    # the cell comes from the universe's full dimensions or from dimensions=
    s6 = S.StructureFactor(u.atoms, n_points=6, q_max=q_max, verbose=False,
                           reciprocal="cell", dimensions=np.asarray(dims, np.float32))
    assert np.array_equal(s6._wavevectors, s._wavevectors)


def test_explicit_wavevectors_are_mapped_to_fractional_space():
    dims = CELLS["truncated_octahedron"]
    u = _universe(dims)
    h = triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float64)
    bstar = 2 * np.pi * np.linalg.inv(h).T
    n = np.array([[0, 0, 0], [1, 0, 0], [0, 3, 1], [2, 5, 7], [11, 0, 4]])
    mk = lambda wv: S.StructureFactor(u.atoms, wavevectors=wv, verbose=False,  # noqa: E731
                                      reciprocal="cell")
    s = mk(n @ bstar)
    assert np.array_equal(s._lattice_n, n)
    np.testing.assert_allclose(s._kvectors, 2 * np.pi * n, atol=1e-12)
    np.testing.assert_allclose(s._wavevectors, n @ bstar, rtol=0, atol=0)
    # negative or off-lattice rows: the general kernel with k = q H^T
    for bad in (np.vstack((n, [[-1, 2, 0]])) @ bstar,
                np.vstack((n @ bstar, [[0.3, 0.1, 0.2]]))):
        s = mk(bad)
        assert s._lattice_n is None and s._lattice_b is None
        np.testing.assert_allclose(s._kvectors, bad @ h.T, rtol=1e-15)
    # the edges mode keeps its own rule (the lattice of the edge lengths)
    e = S.StructureFactor(u.atoms, wavevectors=n @ bstar, verbose=False)
    assert e._lattice_n is None and e._kvectors is e._wavevectors


def test_invalid_arguments():
    u = _universe(CELLS["hexagonal"])
    with pytest.raises(ValueError, match="reciprocal"):
        S.StructureFactor(u.atoms, verbose=False, reciprocal="lattice")
    with pytest.raises(ValueError, match="Invalid unit cell"):
        S.StructureFactor(u.atoms, verbose=False, reciprocal="cell",
                          dimensions=(9.0, 9.0, 9.0, 90.0, 150.0, 150.0))
    with pytest.raises(ValueError, match="Invalid unit cell"):
        S.StructureFactor(u.atoms, verbose=False, reciprocal="cell",
                          dimensions=(9.0, -1.0, 9.0))
    with pytest.raises(ValueError, match="n_surfaces"):
        S.StructureFactor(u.atoms, verbose=False, reciprocal="cell", n_points=4,
                          n_surfaces=2)
    # a cubic orthorhombic cell keeps n_surfaces
    c = _universe((9.0, 9.0, 9.0, 90.0, 90.0, 90.0))
    S.StructureFactor(c.atoms, verbose=False, reciprocal="cell", n_points=4, n_surfaces=2)
    with pytest.raises(ValueError, match="length 3"):
        S.StructureFactor(u.atoms, verbose=False, dimensions=CELLS["hexagonal"])
    with pytest.raises(ValueError, match="length 3 or 6"):
        S.StructureFactor(u.atoms, verbose=False, reciprocal="cell", dimensions=(9.0, 9.0))
    # the ISF inherits the keyword
    i = S.IntermediateScatteringFunction(u.atoms, verbose=False, reciprocal="cell",
                                         n_points=4)
    assert i._cell is not None


def test_set_cell_reports_argument_errors_without_a_device():
    L = _lib.lib()
    assert L.mdh_sq_set_cell(None, None) == _lib.MDH_EINVAL
    assert b"context is NULL" in L.mdh_last_error()


# ---- the fp64 map r -> s = r H^-1 ---------------------------------------------------------

def frac_f64(r, h):
    """tri_frac restated in numpy fp64 (every operation rounded once, the device's order)."""
    x, y, z = (np.asarray(r[:, k], np.float64) for k in range(3))
    ax, bx, by, cx, cy, cz = (float(h[i, j]) for i, j in
                              ((0, 0), (1, 0), (1, 1), (2, 0), (2, 1), (2, 2)))
    sc = z / cz
    sb = (y - sc * cy) / by
    sa = ((x - sb * bx) - sc * cx) / ax
    return np.stack((sa, sb, sc), axis=1)


def frac_exact(r, h):
    """s in longdouble (unit roundoff 2^-64)."""
    x, y, z = (np.asarray(r[:, k]).astype(LD) for k in range(3))
    H = np.asarray(h, np.float64).astype(LD)
    sc = z / H[2, 2]
    sb = (y - sc * H[2, 1]) / H[1, 1]
    sa = ((x - sb * H[1, 0]) - sc * H[2, 0]) / H[0, 0]
    return np.stack((sa, sb, sc), axis=1)


def frac_bound(r, h):
    """Per particle and axis, the bound DESIGN.md 4.3c states for |s~ - s|: the rounding of
    each step of the substitution (2^-53 of the bound on its result) carried forward to
    first order, doubled for the second-order terms -- tri_grid_plan's bound with the
    coordinates' own magnitudes in place of the wrapped cell's."""
    X, Y, Z = (np.abs(np.asarray(r[:, k], np.float64)) for k in range(3))
    ax, bx, by, cx, cy, cz = (abs(float(h[i, j])) for i, j in
                              ((0, 0), (1, 0), (1, 1), (2, 0), (2, 1), (2, 2)))
    Bc = Z / cz * (1 + U); ec = U * Bc                                         # noqa: E702
    Bp1 = Bc * cy * (1 + U); ep1 = cy * ec + U * Bp1                           # noqa: E702
    Bt = (Y + Bp1) * (1 + U); et = ep1 + U * Bt                                # noqa: E702
    Bb = Bt / by * (1 + U); eb = et / by + U * Bb                              # noqa: E702
    Bq1 = Bb * bx * (1 + U); eq1 = bx * eb + U * Bq1                           # noqa: E702
    Br1 = (X + Bq1) * (1 + U); er1 = eq1 + U * Br1                             # noqa: E702
    Bq2 = Bc * cx * (1 + U); eq2 = cx * ec + U * Bq2                           # noqa: E702
    Br2 = (Br1 + Bq2) * (1 + U); er2 = er1 + eq2 + U * Br2                     # noqa: E702
    Ba = Br2 / ax * (1 + U); ea = er2 / ax + U * Ba                            # noqa: E702
    return 2 * np.stack((ea, eb, ec), axis=1)


@pytest.mark.parametrize("name", sorted(CELLS))
@pytest.mark.parametrize("where", ["inside", "far", "float64"])
def test_fractional_map_stays_within_its_bound(name, where):
    rng = np.random.default_rng(7)
    h = triclinic_vectors(np.asarray(CELLS[name], np.float32))
    n = 20000
    f = rng.random((n, 3)) * 2 - 0.5
    if where == "far":                      # many cells away, either side
        f += rng.integers(-5000, 5000, (n, 3))
    r = f @ h.astype(np.float64)
    if where != "float64":
        r = r.astype(np.float32)
    got = frac_f64(r, h)
    want = frac_exact(r, h)
    err = np.abs((got.astype(LD) - want).astype(np.float64))
    bound = frac_bound(r, h)
    assert np.all(err <= bound), float((err / bound).max())
    # the bound is a few ulps of the magnitudes involved, not a loose cap
    assert np.all(bound <= 64 * U * (np.abs(got) + np.abs(r).max(axis=1)[:, None]
                                     / np.diag(h).min()))
