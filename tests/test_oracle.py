"""CPU: the oracle against the golden fixtures (generated from the real reference)."""
import numpy as np
import pytest

from conftest import universe_from
from oracle import ref_harness, reference_port as rp

RDF_CASES = ["lj1000", "twogroup", "excl11", "excl410", "dropz", "dropx_density",
             "lattice_edges", "noncubic_npt", "unwrapped"]


def rdf_kwargs(g):
    kw = dict(n_bins=int(g["n_bins"]), range=tuple(float(x) for x in g["range"]))
    if "exclusion" in g:
        kw["exclusion"] = tuple(int(x) for x in g["exclusion"])
    if "drop_axis" in g:
        kw["drop_axis"] = int(g["drop_axis"])
    return kw


def rdf_groups(u, g):
    if "n_cat" in g:
        n = int(g["n_cat"])
        return u.select(slice(0, n)), u.select(slice(n, u.atoms.n_atoms))
    return u.atoms, None


def test_kat_radial_histogram(golden):
    """The reference's own known-answer construction
    (tests/test_analysis_structure.py:21-40) pins the restated distances."""
    g = golden("kat_radial_histogram")
    got = rp.radial_histogram(g["origin"], g["neighbors"], int(g["n_bins"]),
                              tuple(g["range"]), g["dims"])
    assert np.array_equal(got, g["reference_counts"])
    assert np.array_equal(got, g["expected_from_norms"])


@pytest.mark.parametrize("name", RDF_CASES)
def test_rdf_port_matches_golden(golden, name):
    g = golden(f"rdf_{name}")
    u = universe_from(g)
    ag1, ag2 = rdf_groups(u, g)
    kw = rdf_kwargs(g)
    if name == "dropx_density":
        kw["norm"] = "density"
    out = rp.rdf_run(u, ag1, ag2, **kw)
    assert np.array_equal(out["counts"], g["counts"])
    np.testing.assert_allclose(out["rdf"], g["rdf"], rtol=1e-6)


@pytest.mark.parametrize("name", ["lj1000", "noncubic_npt", "excl11"])
def test_bruteforce_equals_cells(golden, name):
    """The two oracle search strategies must agree pair for pair."""
    g = golden(f"rdf_{name}")
    pos, dims = g["positions"][0], np.atleast_2d(g["dims"])[0]
    rmax = float(min(g["range"][1], dims[:3].min() / 3.001))
    pb, db = rp.capped_distance(pos, pos, rmax, -1e-16, box=dims, method="bruteforce")
    pc, dc = rp.capped_distance(pos, pos, rmax, -1e-16, box=dims, method="nsgrid")
    ob = np.lexsort((pb[:, 1], pb[:, 0]))
    oc = np.lexsort((pc[:, 1], pc[:, 0]))
    assert np.array_equal(pb[ob], pc[oc])
    assert np.array_equal(db[ob], dc[oc])


def test_sq_port_matches_golden(golden):
    g = golden("sq_small")
    u = universe_from(g)
    n = int(g["n_cat"])
    cat, an = u.select(slice(0, n)), u.select(slice(n, u.atoms.n_atoms))
    for mode in (None, "pair", "partial"):
        out = rp.ssf_run(u, [cat, an], mode=mode, n_points=int(g["n_points"]),
                         q_max=float(g["q_max"]))
        for form in ("exp", "trig"):
            np.testing.assert_allclose(out["ssf"], g[f"ssf_{mode}_{form}"],
                                       rtol=1e-9, atol=1e-12)
            np.testing.assert_allclose(out["wavenumbers"],
                                       g[f"wavenumbers_{mode}_{form}"], rtol=1e-13)
    out = rp.ssf_run(u, [u.atoms], n_points=int(g["n_points"]),
                     q_max=float(g["q_max"]), sort=False, unique=False, n_threads=2)
    np.testing.assert_allclose(out["ssf"], g["ssf_raw"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(out["wavevectors"], g["wavevectors_raw"], rtol=0, atol=0)
    rho = rp.delta_fourier_transform_sum(g["wavevectors_raw"],
                                         g["positions"][-1].astype(np.float64))
    np.testing.assert_allclose(rho, g["rho_last"], rtol=1e-10, atol=1e-9)
    out = rp.ssf_run(u, [cat, an], mode="partial", wavevectors=g["wavevectors_user"],
                     sort=False, unique=False)
    np.testing.assert_allclose(out["ssf"], g["ssf_user"], rtol=1e-9, atol=1e-12)


def test_sq_port_noncubic(golden):
    g = golden("sq_noncubic")
    u = universe_from(g)
    out = rp.ssf_run(u, [u.atoms], n_points=int(g["n_points"]), q_max=float(g["q_max"]))
    np.testing.assert_allclose(out["ssf"], g["ssf"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(out["wavenumbers"], g["wavenumbers"], rtol=1e-13)


@pytest.mark.parametrize("mode", [None, "pair", "partial"])
def test_isf_port_matches_golden(golden, mode):
    """oracle isf_run vs fixtures produced by the reference's real
    IntermediateScatteringFunction (both forms are stored; the port restates form=exp)."""
    g = golden("isf_small")
    u = universe_from(g)
    n = int(g["n_cat"])
    cat, an = u.select(slice(0, n)), u.select(slice(n, u.atoms.n_atoms))
    o = rp.isf_run(u, [cat, an], mode=mode, n_points=int(g["n_points"]),
                   q_max=float(g["q_max"]), n_lags=int(g["n_lags"]), incoherent=True,
                   dt=float(g["dt"]))
    for form in ("exp", "trig"):
        np.testing.assert_allclose(o["cisf"], g[f"cisf_{mode}_{form}"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(o["iisf"], g[f"iisf_{mode}_{form}"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(o["times"], g[f"times_{mode}_exp"])
    np.testing.assert_allclose(o["wavenumbers"], g[f"wavenumbers_{mode}_exp"], rtol=1e-13)
    if mode is None:
        o = rp.isf_run(u, [u.atoms], n_points=int(g["n_points"]), q_max=float(g["q_max"]),
                       incoherent=True, sort=False, unique=False, dt=float(g["dt"]),
                       start=2, stop=14, step=3)
        np.testing.assert_allclose(o["cisf"], g["cisf_strided"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(o["iisf"], g["iisf_strided"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(o["times"], g["times_strided"])
        # F_s(q, 0) = 1 and F(q, 0) = S(q)
        np.testing.assert_allclose(o["iisf"][0], 1.0, rtol=1e-12)
    if mode == "partial":
        # user wavevectors off the lattice, in the order given
        o = rp.isf_run(u, [cat, an], mode=mode, wavevectors=g["wavevectors_user"],
                       n_lags=4, incoherent=True, sort=False, unique=False,
                       dt=float(g["dt"]))
        np.testing.assert_allclose(o["cisf"], g["cisf_user"], rtol=1e-9, atol=1e-10)
        np.testing.assert_allclose(o["iisf"], g["iisf_user"], rtol=1e-9, atol=1e-10)


def test_scsf_port_matches_golden(golden):
    """oracle scsf_run vs fixtures of the reference's real SingleChainStructureFactor."""
    g = golden("scsf_small")
    u = universe_from(g)
    kw = dict(n_points=int(g["n_points"]), n_chains=int(g["n_chains"]),
              n_monomers=int(g["n_monomers"]))
    for unwrap in (False, True):
        o = rp.scsf_run(u, u.atoms, unwrap=unwrap, **kw)
        np.testing.assert_allclose(o["scsf"], g[f"scsf_unwrap{int(unwrap)}"], rtol=1e-12)
        np.testing.assert_allclose(o["wavenumbers"], g["wavenumbers"], rtol=1e-13)
    o = rp.scsf_run(u, u.atoms, start=1, stop=6, step=2, **kw)
    np.testing.assert_allclose(o["scsf"], g["scsf_strided"], rtol=1e-12)
    assert abs(o["scsf"][0] - 20.0) < 1e-12          # S_sc(0) = chain length


@pytest.mark.parametrize("tag", ["equal", "unequal"])
def test_centres_of_mass_match_the_reference(golden, tag):
    """The host centre-of-mass helper (whose operation order the device kernel follows) vs
    the reference's real ``center_of_mass`` (algorithm/molecule.py:15-310; fixture made by
    tests/golden/make_golden.py com): within one fp64 ulp, and identical after the
    rounding to float32 that ``capped_distance`` applies to its inputs."""
    from mdhelper_b200.analysis.structure import _centers_of_mass
    from mdhelper_b200.universe import SyntheticUniverse
    g = golden("com_ref")
    u = SyntheticUniverse(g[f"{tag}_positions"], g[f"{tag}_dims"],
                          resindices=g[f"{tag}_resindices"],
                          segindices=g[f"{tag}_segindices"], masses=g[f"{tag}_masses"])
    for grouping in ("residues", "segments"):
        for f in range(4):
            ts = u.trajectory[f]
            got = _centers_of_mass(u.atoms, grouping, ts.positions)
            want = g[f"{tag}_com_{grouping}"][f]
            np.testing.assert_allclose(got, want, rtol=5e-16)
            assert np.array_equal(got.astype(np.float32), want.astype(np.float32))
    if ref_harness.available():
        # live: the real function on the duck-typed universe gives the stored centres
        import importlib
        ref_harness.load()
        mol = importlib.import_module("mdhelper.algorithm.molecule")
        u.trajectory[2]
        np.testing.assert_array_equal(mol.center_of_mass(u.atoms, "residues"),
                                      g[f"{tag}_com_residues"][2])


def _triclinic_case(seed=5, n=350):
    rng = np.random.default_rng(seed)
    dims = np.array([10.5, 11.25, 12.0, 75.0, 82.0, 64.0], np.float32)
    h = rp.triclinic_vectors(dims).astype(np.float64)
    p = (rng.random((n, 3)) @ h).astype(np.float32)
    return dims, h, p


def test_triclinic_minimum_image_is_the_shortest_image():
    """Restated triclinic path of capped_distance (unpinned against MDAnalysis): the
    distances are the mathematical minimum over lattice images to float32 rounding."""
    dims, h, p = _triclinic_case()
    pairs, d = rp.capped_distance(p, p, 4.0, -1e-16, box=dims)
    P = p.astype(np.float64)
    best = np.full((len(p), len(p)), np.inf)
    for i in range(-2, 3):
        for j in range(-2, 3):
            for k in range(-2, 3):
                D = P[None, :, :] - P[:, None, :] + (i * h[0] + j * h[1] + k * h[2])
                best = np.minimum(best, (D ** 2).sum(-1))
    best = np.sqrt(best)
    assert len(d) == (best <= 4.0).sum()
    np.testing.assert_allclose(d, best[pairs[:, 0], pairs[:, 1]], atol=2e-6)


def test_triclinic_with_right_angles_equals_orthorhombic():
    """Property: a diagonal cell matrix through the triclinic arithmetic gives the counts
    of the orthorhombic arithmetic."""
    import oracle
    rng = np.random.default_rng(8)
    dims = np.array([10.0, 11.0, 12.0, 90, 90, 90], np.float32)
    p = (rng.random((500, 3)) * dims[:3]).astype(np.float32)
    q = (rng.random((300, 3)) * dims[:3] * 3 - dims[:3]).astype(np.float32)     # unwrapped
    h = np.ascontiguousarray(np.diag(dims[:3]), np.float32)
    L = oracle.lib()
    for a, b in ((p, p), (p, q)):
        cap = len(a) * len(b)
        pairs, dist = np.empty((cap, 2), np.int64), np.empty(cap)
        m = L.mdho_capped_distance_triclinic(a.ctypes.data, len(a), b.ctypes.data, len(b),
                                             h.ctypes.data, 5.0, -1e-16, pairs.ctypes.data,
                                             dist.ctypes.data, cap)
        got = np.histogram(dist[:m], bins=80, range=(0, 5.0))[0]
        assert np.array_equal(got, rp.radial_histogram(a, b, 80, (0, 5.0), dims))


def test_triclinic_lattice_translation_invariance():
    """Property: moving particles by lattice vectors changes nothing.  Cell and coordinates
    are dyadic rationals, so the translations are exact in float32."""
    rng = np.random.default_rng(9)
    h = np.array([[8, 0, 0], [2, 8, 0], [-1, 3, 8]], np.float32)
    frac = rng.integers(0, 1024, (260, 3)) / 1024.0
    p = (frac @ h.astype(np.float64)).astype(np.float32)
    shift = rng.integers(-2, 3, (260, 3)).astype(np.float64) @ h.astype(np.float64)
    q = (p.astype(np.float64) + shift).astype(np.float32)
    assert np.array_equal(q.astype(np.float64), p.astype(np.float64) + shift)   # exact
    # dims of that matrix: lengths and angles (the port only needs them to be non-90)
    lx, ly, lz = (np.linalg.norm(h[k].astype(np.float64)) for k in range(3))
    import oracle
    L = oracle.lib()

    def counts(a):
        cap = len(a) ** 2
        pairs, dist = np.empty((cap, 2), np.int64), np.empty(cap)
        m = L.mdho_capped_distance_triclinic(a.ctypes.data, len(a), a.ctypes.data, len(a),
                                             np.ascontiguousarray(h).ctypes.data, 3.9, -1e-16,
                                             pairs.ctypes.data, dist.ctypes.data, cap)
        return np.sort(dist[:m])
    assert np.array_equal(counts(p), counts(q))
    assert lx > 0 and ly > 0 and lz > 0


def test_grid_search_moves_coordinates_into_the_cell_in_float32():
    """Restated `_ortho_pbc` of MDAnalysis' grid search ("parity unpinned"): the port's
    nsgrid path equals brute force over the float32-wrapped copies, the identity for
    coordinates inside the cell, and keeps the known edge cases (-1e-9 -> box)."""
    import oracle
    L = oracle.lib()
    box = np.array([10.0, 11.0, 12.0], np.float32)
    x = np.array([[-1e-9, 5, 13], [25.5, -30.2, 11.999999], [-0.5, 11.0, 0.0],
                  [10.0, -11.0, 24.0]], np.float32)
    y = x.copy()
    L.mdho_ortho_pbc(y.ctypes.data, len(y), box.ctypes.data)
    assert y[0, 0] == np.float32(10.0) and y[0, 2] == np.float32(1.0)
    assert np.all((y >= 0) & (y <= box))
    d = x.astype(np.float64) - y
    np.testing.assert_allclose(d - box * np.round(d / box), 0.0, atol=4e-6)    # same point
    rng = np.random.default_rng(4)
    dims = np.array([10.0, 11.0, 12.0, 90, 90, 90], np.float32)
    inside = (rng.random((300, 3)) * box).astype(np.float32)
    z = inside.copy()
    L.mdho_ortho_pbc(z.ctypes.data, len(z), box.ctypes.data)
    assert np.array_equal(z, inside)
    p = ((rng.random((400, 3)) * 5 - 2) * box).astype(np.float32)
    w = p.copy()
    L.mdho_ortho_pbc(w.ctypes.data, len(w), box.ctypes.data)
    grid = rp.radial_histogram(p, p, 40, (0.0, 3.0), dims, method="nsgrid")
    assert np.array_equal(grid, rp.radial_histogram(w, w, 40, (0.0, 3.0), dims,
                                                    method="bruteforce"))
    # the method rule (SURVEY.md Appendix A item 2): small cut-off -> grid search
    assert np.array_equal(grid, rp.radial_histogram(p, p, 40, (0.0, 3.0), dims))


def test_isf_port_on_float64_centres_matches_the_reference(golden):
    """tests/golden/f64_ref.npz (the reference's real IntermediateScatteringFunction with
    groupings="residues"): the port's sliding window, fed the float64 centres of mass of
    the residues, reproduces it -- the checker of the GPU path that keeps those centres
    in float64."""
    from mdhelper_b200.universe import SyntheticUniverse

    class Centres:
        def __init__(self, group):
            self._g = group
            _, self._inv = np.unique(group.resindices, return_inverse=True)
            self._m = np.asarray(group.masses, dtype=np.float64)
            self.n_atoms = int(self._inv.max()) + 1

        @property
        def positions(self):
            p = np.asarray(self._g.positions, dtype=np.float64)
            out = np.zeros((self.n_atoms, 3))
            np.add.at(out, self._inv, self._m[:, None] * p)
            return out / np.bincount(self._inv, weights=self._m)[:, None]

    g = golden("f64_ref")
    u = SyntheticUniverse(g["isf_positions"], g["isf_dims"], resindices=g["isf_resindices"],
                          masses=g["isf_masses"])
    n_a, n = int(g["isf_n_a"]), u.atoms.n_atoms
    a, b = u.select(slice(0, n_a)), u.select(slice(n_a, n))
    o = rp.isf_run(u, [Centres(a), Centres(b)], mode="partial", n_points=5, n_lags=4,
                   incoherent=True, dt=1.0, n_threads=2)
    np.testing.assert_allclose(o["wavenumbers"], g["isf_wavenumbers"], rtol=1e-12)
    np.testing.assert_allclose(o["cisf"], g["isf_cisf"], rtol=1e-10, atol=1e-11)
    np.testing.assert_allclose(o["iisf"], g["isf_iisf"], rtol=1e-10, atol=1e-11)
