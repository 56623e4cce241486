"""GPU: S(q) and F(q, t) on the reciprocal lattice of triclinic cells (reciprocal="cell",
mdh_sq_set_cell) against the restated reference on the Cartesian wavevectors, the general
kernel, an extended-precision direct sum and crystal physics."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CELLS = {
    "monoclinic": (9.0, 10.0, 11.0, 90.0, 104.0, 90.0),
    "hexagonal": (9.0, 9.0, 12.0, 90.0, 90.0, 120.0),
    "rhombic_dodecahedron": (10.0, 10.0, 10.0, 60.0, 60.0, 90.0),
    "truncated_octahedron": (10.0, 10.0, 10.0, 70.53, 109.47, 70.53),
}
KERNELS = ("lattice_dmma", "lattice_fp64", "general_fp64")


def _S():
    from mdhelper_b200.analysis import structure
    return structure


def _rp():
    from oracle import reference_port as rp
    return rp


def _h(dims):
    from mdhelper_b200.analysis._triclinic import triclinic_vectors
    return triclinic_vectors(np.asarray(dims, np.float32))


def _positions(dims_list, n, seed, lo=-0.5, hi=1.5):
    """float32 coordinates of fractional coordinates in [lo, hi) of each frame's cell."""
    rng = np.random.default_rng(seed)
    dims = np.array(dims_list, np.float32)
    pos = np.empty((len(dims), n, 3), np.float32)
    for f, d in enumerate(dims):
        pos[f] = ((rng.random((n, 3)) * (hi - lo) + lo) @ _h(d).astype(np.float64))
    return pos, dims


def _universe(dims, n=300, frames=3, seed=1, **kw):
    from mdhelper_b200.universe import SyntheticUniverse
    pos, d = _positions([dims] * frames, n, seed)
    return SyntheticUniverse(pos, d[0], **kw)


def _groups(u, split=120):
    return [u.select(slice(0, split)), u.select(slice(split, u.atoms.n_atoms))]


@pytest.mark.parametrize("name", sorted(CELLS))
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("form", ["exp", "trig"])
@pytest.mark.parametrize("mode", [None, "pair", "partial"])
def test_structure_factor_matches_the_reference_on_the_cell_grid(name, kernel, form, mode):
    u = _universe(CELLS[name], seed=len(name))
    g = _groups(u)
    s = _S().StructureFactor(g, mode=mode, form=form, n_points=6, q_max=2.5, kernel=kernel,
                             reciprocal="cell", verbose=False).run()
    assert s._ctx.sq_kernel() == kernel
    want = _rp().ssf_run(u, g, mode=mode, wavevectors=s._wavevectors)
    np.testing.assert_array_equal(s.results.wavenumbers, want["wavenumbers"])
    np.testing.assert_allclose(s.results.ssf, want["ssf"], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name", sorted(CELLS))
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("mode", [None, "partial"])
def test_isf_matches_the_reference_on_the_cell_grid(name, kernel, mode):
    u = _universe(CELLS[name], n=200, frames=7, seed=3)
    g = _groups(u, 80)
    want = None
    for batch in (1, 3, 7):
        i = _S().IntermediateScatteringFunction(
            g, mode=mode, n_points=5, q_max=2.0, n_lags=4, incoherent=True, kernel=kernel,
            reciprocal="cell", batch_frames=batch, verbose=False).run()
        assert i._ctx.sq_kernel() == kernel
        if want is None:
            want = _rp().isf_run(u, g, mode=mode, wavevectors=i._wavevectors, n_lags=4,
                                 incoherent=True)
        np.testing.assert_array_equal(i.results.wavenumbers, want["wavenumbers"])
        np.testing.assert_allclose(i.results.cisf, want["cisf"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(i.results.iisf, want["iisf"], rtol=1e-9, atol=1e-12)
        if mode is None:
            np.testing.assert_allclose(i.results.iisf[0], 1.0, rtol=1e-12)
    # F(q, 0) = S(q) over the same frames
    s = _S().StructureFactor(g, mode=mode, n_points=5, q_max=2.0, kernel=kernel,
                             reciprocal="cell", verbose=False).run()
    np.testing.assert_allclose(i.results.cisf[0], s.results.ssf, rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name", sorted(CELLS))
def test_lattice_kernels_equal_the_general_kernel_on_cartesian_wavevectors(name):
    import _sq_reference as R
    u = _universe(CELLS[name], n=500, frames=2, seed=5)
    c = _S().StructureFactor(u.atoms, n_points=7, q_max=3.0, reciprocal="cell",
                             unique=False, sort=False, verbose=False).run()
    assert c._ctx.sq_kernel() in ("lattice_dmma", "lattice_fp64")
    e = _S().StructureFactor(u.atoms, wavevectors=c._wavevectors, unique=False, sort=False,
                             verbose=False).run()
    assert e._ctx.sq_kernel() == "general_fp64"
    np.testing.assert_allclose(c.results.ssf, e.results.ssf, rtol=1e-9, atol=1e-12)
    # rho(q) of the last frame against a longdouble direct sum on longdouble s = r H^-1
    r = u.trajectory[1].positions.astype(np.longdouble)
    H = _h(CELLS[name]).astype(np.float64).astype(np.longdouble)
    sc = r[:, 2] / H[2, 2]
    sb = (r[:, 1] - sc * H[2, 1]) / H[1, 1]
    sa = ((r[:, 0] - sb * H[1, 0]) - sc * H[2, 0]) / H[0, 0]
    s = np.stack((sa, sb, sc), axis=1)
    want = R.rho_ref(s, c._lattice_n, np.full(3, 2 * np.pi))
    got = c._ctx.sq_fetch_rho()[0]
    np.testing.assert_allclose(got, want.astype(np.complex128), rtol=0, atol=1e-9 * len(r))


@pytest.mark.parametrize("name", sorted(CELLS))
def test_perfect_crystal_has_bragg_peaks_at_multiples_of_m(name):
    from mdhelper_b200.universe import SyntheticUniverse
    m = 4
    d = np.array(CELLS[name], np.float64)
    dims = np.array([*(d[:3] * m), *d[3:]], np.float32)
    H = _h(dims).astype(np.float64) / m                  # the primitive cell
    ijk = np.stack(np.meshgrid(*3 * [np.arange(m)], indexing="ij"), -1).reshape(-1, 3)
    pos = (ijk @ H).astype(np.float32)[None]
    u = SyntheticUniverse(pos, dims)
    s = _S().StructureFactor(u.atoms, n_points=9, reciprocal="cell", unique=False,
                             sort=False, verbose=False).run()
    N = len(ijk)
    n = s._lattice_n
    want = np.where(np.all(n % m == 0, axis=1), float(N), 0.0)
    np.testing.assert_allclose(s.results.ssf[0], want, rtol=0, atol=1e-9 * N)


def _ctx_ssf(pos, H, lattice_n, kernel="auto"):
    from mdhelper_b200 import _lib
    ctx = _lib.Context(0)
    F, n = pos.shape[:2]
    ctx.sq_configure(n, [0, n], 2 * np.pi * lattice_n, [(-1, -1)], lattice_n=lattice_n,
                     lattice_b=np.full(3, 2 * np.pi), mode=kernel)
    ctx.sq_set_cell(H)
    p = np.ascontiguousarray(pos)
    ctx.sq_accumulate(p, 3 * n, F, f64=p.dtype == np.float64)
    return ctx.sq_fetch()[0]


def test_two_bases_of_one_lattice_give_the_same_s():
    rng = np.random.default_rng(11)
    H = _h(CELLS["truncated_octahedron"]).astype(np.float64)
    Um = np.array([[1, 0, 0], [1, 1, 0], [-1, 2, 1]], np.float64)   # unimodular, lower
    H2 = Um @ H                                                       # still lower triangular
    pos = (rng.random((2, 400, 3)) * 2 - 0.5) @ H
    n1 = np.stack(np.meshgrid(*3 * [np.arange(6)], indexing="ij"), -1).reshape(-1, 3)
    # B2* = 2 pi (U H)^-T = U^-T B1*, so q = n1 B1* = n2 B2* for n2 = n1 U^T
    n2 = n1 @ Um.T.astype(np.int64)
    both = np.all((n2 >= 0) & (n2 < 40), axis=1)
    assert both.sum() > 30
    s1 = _ctx_ssf(pos, H, n1[both].astype(np.int32))
    s2 = _ctx_ssf(pos, H2, n2[both].astype(np.int32))
    np.testing.assert_allclose(s1, s2, rtol=1e-9, atol=1e-9 * 400)


@pytest.mark.parametrize("kernel", KERNELS)
def test_moving_particles_by_cell_vectors_leaves_s_unchanged(kernel):
    rng = np.random.default_rng(12)
    # dyadic cell and coordinates: the moved coordinates are exact in float32
    H = np.array([[8.0, 0, 0], [2.5, 7.75, 0], [-1.25, 3.5, 6.5]])
    pos = (np.round(rng.random((2, 500, 3)) @ H * 1024) / 1024).astype(np.float32)
    shift = rng.integers(-20, 21, (2, 500, 3)) @ H
    moved = (pos + shift).astype(np.float32)
    assert np.array_equal(moved.astype(np.float64), pos + shift)
    n = np.stack(np.meshgrid(*3 * [np.arange(7)], indexing="ij"), -1).reshape(-1, 3)
    n = n.astype(np.int32)
    a, b = _ctx_ssf(pos, H, n, kernel), _ctx_ssf(moved, H, n, kernel)
    np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-9 * 500)


def test_npt_trajectory_matches_the_reference():
    from mdhelper_b200.universe import SyntheticUniverse
    base = np.array(CELLS["rhombic_dodecahedron"], np.float64)
    dims = [np.array([*(base[:3] * (1 + 0.02 * f)), *base[3:]]) for f in range(4)]
    pos, d = _positions(dims, 300, 4)
    u = SyntheticUniverse(pos, d)
    s = _S().StructureFactor(u.atoms, n_points=6, q_max=2.5, reciprocal="cell",
                             verbose=False).run()
    want = _rp().ssf_run(u, [u.atoms], wavevectors=s._wavevectors)
    np.testing.assert_allclose(s.results.ssf, want["ssf"], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("host_com", [False, True])
def test_residue_centres_match_a_float64_direct_sum(host_com):
    n_res, per = 150, 3
    u = _universe(CELLS["monoclinic"], n=n_res * per, frames=3, seed=6,
                  resindices=np.repeat(np.arange(n_res), per),
                  masses=np.tile([12.0, 1.0, 16.0], n_res))
    s = _S().StructureFactor(u.atoms, groupings="residues", n_points=6, q_max=2.5,
                             reciprocal="cell", host_com=host_com, unique=False, sort=False,
                             verbose=False).run()
    m = np.tile([12.0, 1.0, 16.0], n_res)
    want = np.zeros(len(s._wavevectors))
    for f in range(3):
        r = u.trajectory[f].positions.astype(np.float64) * m[:, None]
        com = r.reshape(n_res, per, 3).sum(axis=1) / m[:per].sum()
        rho = _rp().delta_fourier_transform_sum(s._wavevectors, com)
        want += (rho * rho.conj()).real
    np.testing.assert_allclose(s.results.ssf[0], want / (3 * n_res), rtol=1e-9, atol=1e-12)


def test_orthorhombic_cell_mode_is_the_edges_mode():
    u = _universe((9.0, 10.0, 11.0, 90.0, 90.0, 90.0), n=400)
    for cls, kw in ((_S().StructureFactor, {}),
                    (_S().IntermediateScatteringFunction, dict(incoherent=True, n_lags=2))):
        e = cls(u.atoms, n_points=6, verbose=False, **kw).run()
        c = cls(u.atoms, n_points=6, verbose=False, reciprocal="cell", **kw).run()
        for k, v in e.results.items():
            if isinstance(v, np.ndarray):
                assert np.array_equal(c.results[k], v), k


def test_combined_analysis_and_file_reader_equal_separate_runs(tmp_path):
    from conftest import file_universe
    from mdhelper_b200.analysis import CombinedAnalysis
    dims = CELLS["truncated_octahedron"]
    u = _universe(dims, n=600, frames=5, seed=9)
    mk_r = lambda: _S().RadialDistributionFunction(u.atoms, n_bins=40, range=(0.0, 4.0),  # noqa
                                                   verbose=False)
    mk_s = lambda uu: _S().StructureFactor(uu.atoms, n_points=6, q_max=2.5,  # noqa: E731
                                           reciprocal="cell", verbose=False)
    r0, s0 = mk_r().run(), mk_s(u).run()
    r1, s1 = mk_r(), mk_s(u)
    CombinedAnalysis(r1, s1, batch_frames=2).run()
    assert np.array_equal(r1.results.counts, r0.results.counts)
    np.testing.assert_allclose(s1.results.ssf, s0.results.ssf, rtol=1e-12)
    pos = np.stack([u.trajectory[f].positions for f in range(5)])
    uf = file_universe(tmp_path, pos, np.asarray(dims, np.float32))
    sf = mk_s(uf).run()
    np.testing.assert_allclose(sf.results.ssf, s0.results.ssf, rtol=1e-12)


def test_set_cell_errors():
    from mdhelper_b200 import _lib
    ctx = _lib.Context(0)
    H = _h(CELLS["hexagonal"]).astype(np.float64)
    with pytest.raises(RuntimeError, match="mdh_sq_configure"):
        ctx.sq_set_cell(H)                                   # MDH_ESTATE
    n = np.array([[0, 0, 0], [1, 2, 3]], np.int32)
    ctx.sq_configure(4, [0, 4], 2 * np.pi * n, [(-1, -1)], lattice_n=n,
                     lattice_b=np.full(3, 2 * np.pi))
    for bad, what in (((0, 0), "valid cell"), ((1, 1), "valid cell"), ((2, 2), "valid cell"),
                      ((1, 1), "finite"), ((0, 1), "lower triangular")):
        h = H.copy()
        h[bad] = -1.0 if what == "valid cell" else np.nan if what == "finite" else 1.0
        with pytest.raises(ValueError, match=what):
            ctx.sq_set_cell(h)
    ctx.sq_set_cell(H)
    ctx.sq_set_cell(None)
