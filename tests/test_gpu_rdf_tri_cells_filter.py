"""GPU: the fp32 filter of the triclinic cell list (rdf_tri_cells_filter_kernel) gives the
counts of the fp64 cell list (arith "off"), of the all-pairs kernel and of the restated
reference (the CPU oracle of _threshold_pairs), bit for bit; the audit finds no certified
candidate in a wrong bin; declined frames are counted exactly."""
import numpy as np
import pytest

from _threshold_pairs import tri_ref_d2

pytestmark = pytest.mark.gpu

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)              # rhombic dodecahedron
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)          # truncated octahedron
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)           # strongly tilted monoclinic
HEX = (1.0, 1.0, 1.0, 90.0, 90.0, 120.0)            # hexagonal


def _cell(dims):
    from oracle import reference_port as rp
    return rp.triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float32)


def _scaled(shape, L):
    return np.array([L * shape[0], L * shape[1], L * shape[2], *shape[3:]], np.float32)


def _width(h):
    h = h.astype(np.float64)
    vol = abs(np.linalg.det(h))
    a, b, c = h
    return min(vol / np.linalg.norm(np.cross(b, c)), vol / np.linalg.norm(np.cross(c, a)),
               vol / np.linalg.norm(np.cross(a, b)))


def _fluid(n, h, rng, lo=0.0, hi=1.0):
    return ((rng.random((n, 3)) * (hi - lo) + lo) @ h.astype(np.float64)).astype(np.float32)


def _run(p, cells, n_bins, rng_, arith, mode="cells", *, q=None, exclusion=None, device=False,
         drop_axis=None):
    import torch
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    F, n = p.shape[:2]
    m = n if q is None else q.shape[1]
    ctx = _lib.Context(0)
    try:
        ctx.rdf_set_filter(arith)
        ctx.rdf_configure(n, m, q is None, squared_thresholds(n_bins, rng_), rng_[0], rng_[1],
                          mode=mode, exclusion=exclusion, drop_axis=drop_axis)
        a, b = p, (p if q is None else q)
        if device:
            a = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            b = a if q is None else torch.from_numpy(np.ascontiguousarray(b)).cuda()
        ctx.rdf_accumulate_triclinic(a, 3 * n, b, 3 * m, cells, F, device=device)
        return ctx.rdf_fetch(), ctx.rdf_filter_stats(), ctx.rdf_pair_evaluations()
    finally:
        ctx.close()


def _oracle(p, cells, n_bins, rng_, *, q=None, exclusion=None, drop_axis=None):
    """Counts of every ordered pair from the reference's 27-image fp64 arithmetic."""
    from mdhelper_b200.analysis._binning import squared_thresholds
    thr = squared_thresholds(n_bins, rng_)
    out = np.zeros(n_bins, np.int64)
    for f in range(p.shape[0]):
        a = p[f].copy()
        b = a if q is None else q[f].copy()
        if drop_axis is not None:
            a[:, drop_axis] = 0.0
            b[:, drop_axis] = 0.0
        for i0 in range(0, len(a), 500):
            i, j = np.meshgrid(np.arange(i0, min(i0 + 500, len(a))), np.arange(len(b)),
                               indexing="ij")
            i, j = i.ravel(), j.ravel()
            if exclusion is not None:
                keep = i // exclusion[0] != j // exclusion[1]
                i, j = i[keep], j[keep]
            d2 = tri_ref_d2(a[i], b[j], cells[f])
            k = np.searchsorted(thr, d2, side="right") - 1
            k = k[(k >= 0) & (k < n_bins)]
            out += np.bincount(k, minlength=n_bins)
    return out


def _check(p, cells, n_bins, rng_, *, oracle=True, declined=0, **kw):
    got, st, ev = _run(p, cells, n_bins, rng_, "auto", **kw)
    off, st_off, ev_off = _run(p, cells, n_bins, rng_, "off", **kw)
    aud, st_aud, _ = _run(p, cells, n_bins, rng_, "audit", **kw)
    assert got.sum() > 0
    assert np.array_equal(got, off), kw
    assert np.array_equal(aud, off), kw
    allp, _, _ = _run(p, cells, n_bins, rng_, "off", "allpairs", **kw)
    assert np.array_equal(got, allp), kw
    if oracle:
        want = _oracle(p, cells, n_bins, rng_, q=kw.get("q"), exclusion=kw.get("exclusion"),
                       drop_axis=kw.get("drop_axis"))
        assert np.array_equal(got, want), kw
    F = p.shape[0]
    assert st_aud["audit_violations"] == 0, st_aud
    assert st["triclinic_frames"] == F - declined and st["declined_frames"] == declined, st
    assert st_aud["triclinic_frames"] == F - declined
    assert st_off["triclinic_frames"] == 0 and st_off["declined_frames"] == 0
    # the same runs as the fp64 cell list: the same candidate count
    assert ev == ev_off
    return st, st_aud


@pytest.mark.parametrize("dims", [(10.5, 11.25, 12.0, 75.0, 82.0, 64.0),
                                  (10.0, 11.5, 12.5, 90.0, 90.0, 70.0),
                                  (11.0, 11.0, 11.0, 60.0, 60.0, 60.0),
                                  _scaled(RD, 12.0), _scaled(TO, 12.0), _scaled(TILT, 12.0),
                                  _scaled(HEX, 12.0)], ids=range(7))
def test_oracle_cells_one_and_two_groups(dims):
    rng = np.random.default_rng(int(sum(dims)))
    h = _cell(dims)
    cells = np.stack([h, h])
    r_hi = _width(h) / 3.3
    p = np.stack([_fluid(1800, h, rng, -2.0, 3.0), _fluid(1800, h, rng)])
    _check(p, cells, 70, (0.0, r_hi))
    q = np.stack([_fluid(900, h, rng), _fluid(900, h, rng, -1.0, 2.0)])
    _check(p, cells, 70, (0.4 * r_hi, r_hi), q=q)


@pytest.mark.parametrize("exclusion", [(1, 1), (4, 10)])
def test_exclusions(exclusion):
    rng = np.random.default_rng(2)
    h = _cell(_scaled(TO, 14.0))
    r_hi = _width(h) / 3.2
    p = _fluid(2000, h, rng)[None]
    q = None
    if exclusion[0] != exclusion[1]:
        q = _fluid(5000, h, rng)[None]
    _check(p, h[None], 50, (0.0, r_hi), exclusion=exclusion, q=q)
    _check(p, h[None], 50, (0.3 * r_hi, r_hi), exclusion=exclusion, q=q)


def _lattice(h, r_hi, edges, rng):
    """Particles at cell faces and corners (+- ulps, 1 - ulp) and partners at the bin
    edges, at r_hi and next to them, pointing out of the cell."""
    hd = h.astype(np.float64)
    one_m = np.nextafter(1.0, 0.0)
    spots = [0.0, 1e-6, 0.01, 0.5, 0.99, one_m]
    lengths = np.concatenate([[r_hi * (1 - 1e-7), r_hi, r_hi * (1 + 1e-7)], edges[1:-1],
                              edges[1:-1] * (1 + 1e-7), edges[1:-1] * (1 - 1e-7)])
    first, second = [], []
    for fa in spots:
        for fb in spots:
            for fc in spots:
                fr = np.array([fa, fb, fc])
                base = fr @ hd
                for _ in range(3):
                    sgn = np.where(fr > 0.5, 1.0, np.where(fr < 0.5, -1.0, rng.choice([-1, 1], 3)))
                    v = np.abs(rng.normal(size=3)) * sgn
                    v /= np.linalg.norm(v)
                    first.append(base)
                    second.append(base + v * rng.choice(lengths))
    return np.concatenate([first, second]).astype(np.float32)


@pytest.mark.parametrize("shape", [RD, TO, TILT, HEX])
def test_adversarial_lattices_on_bin_edges(shape):
    h = _cell(_scaled(shape, 9.0))
    r_hi = _width(h) / 3.05
    edges = np.linspace(0.0, r_hi, 41)
    p = _lattice(h, r_hi, edges, np.random.default_rng(5))[None]
    _check(p, h[None], 40, (0.0, r_hi))
    _check(p, h[None], 40, (0.2 * r_hi, r_hi), q=p[:, ::-1].copy())


def test_many_bins_and_lower_edge():
    rng = np.random.default_rng(3)
    h = _cell(_scaled(RD, 16.0))
    r_hi = _width(h) / 3.1
    p = _fluid(3000, h, rng)[None]
    _check(p, h[None], 1000, (0.0, r_hi), oracle=False)
    _check(p, h[None], 1000, (0.5, r_hi))


def test_flat_grid_drop_axis_2():
    rng = np.random.default_rng(4)
    for shape in (HEX, TILT):
        dims = _scaled(shape, 14.0)
        dims[2] = 20.0
        h = _cell(dims)
        p = _fluid(2500, h, rng)[None]
        r_hi = 14.0 / 3.3 * 0.8
        _check(p, h[None], 40, (0.0, r_hi), drop_axis=2)


def test_unwrapped_host_and_device():
    rng = np.random.default_rng(5)
    h = _cell(_scaled(TILT, 14.0))
    r_hi = _width(h) / 3.2
    p = np.stack([_fluid(2000, h, rng, -2.0, 3.0), _fluid(2000, h, rng, -1.0, 1.0)])
    cells = np.stack([h, h])
    _check(p, cells, 40, (0.0, r_hi))
    _check(p, cells, 40, (0.0, r_hi), device=True, oracle=False)
    q = np.stack([_fluid(800, h, rng, -1.0, 2.0), _fluid(800, h, rng)])
    _check(p, cells, 40, (0.0, r_hi), q=q, device=True, oracle=False)


def test_quirk_of_the_27_images_in_a_truncated_octahedron():
    """Candidates whose image m' is not among the reference's 27 are not counted, even
    when their true distance is in range."""
    rng = np.random.default_rng(7)
    h = _cell(_scaled(TO, 13.0))
    hd = h.astype(np.float64)
    r_hi = _width(h) / 3.05
    p = _fluid(2000, h, rng)[None]
    # m' = (2, -1, 1): the shortest image of dx is u = dx - (2a - b + c)
    u = np.array([-0.6 * r_hi, 0.1, -0.1])
    dxq = u + 2 * hd[0] - hd[1] + hd[2]
    for k in range(20):
        wi = np.array([0.05, 0.5 * hd[1, 1], 0.05]) + 0.05 * rng.random(3)
        p[0, 2 * k] = wi
        p[0, 2 * k + 1] = wi + dxq + 0.02 * rng.random(3)
    _check(p, h[None], 60, (0.0, r_hi))


def test_declined_frames():
    """A frame with NaN coordinates and a far frame are declined on the device and
    counted exactly; the cell matrix alone leaves every frame eligible."""
    rng = np.random.default_rng(8)
    h = _cell(_scaled(RD, 14.0))
    r_hi = _width(h) / 3.2
    p = np.stack([_fluid(2000, h, rng) for _ in range(3)])
    p[1, 7] = [np.nan, 1.0, 1.0]
    p[2, 9] = [1.0e20, -3.0e19, 5.0e19]            # far: the wrap cannot bring it back
    cells = np.stack([h, h, h])
    got, st, ev = _run(p, cells, 40, (0.0, r_hi), "auto")
    off, _, ev_off = _run(p, cells, 40, (0.0, r_hi), "off")
    allp, _, _ = _run(p, cells, 40, (0.0, r_hi), "off", "allpairs")
    assert np.array_equal(got, off) and np.array_equal(got, allp)
    assert st["triclinic_frames"] == 1 and st["declined_frames"] == 2 and ev == ev_off
    aud, st_aud, _ = _run(p, cells, 40, (0.0, r_hi), "audit")
    assert np.array_equal(aud, off) and st_aud["audit_violations"] == 0
    # the window of the cell matrix agrees with the kernel's choice
    from mdhelper_b200 import _lib
    win = _lib.triclinic_cells_filter_window(40, 0.0, r_hi, cells)
    assert all(w["eligible"] == 1 for w in win)


def test_mixed_orthorhombic_and_triclinic_trajectory():
    from mdhelper_b200.universe import SyntheticUniverse
    from mdhelper_b200.analysis import structure as S
    from oracle import reference_port as rp
    rng = np.random.default_rng(6)
    n, L = 4000, 17.0
    dims = np.array([[L, L, L, 60, 60, 90], [L, L, L, 90, 90, 90],
                     [L, L, L, 70.53, 109.47, 70.53]], np.float32)
    pos = np.stack([_fluid(n, _cell(d), rng) for d in dims])
    u = SyntheticUniverse(pos, dims)
    kw = dict(n_bins=50, range=(0.0, 2.5), verbose=False, mode="cells")
    auto = S.RadialDistributionFunction(u.atoms, **kw).run()
    off = S.RadialDistributionFunction(u.atoms, arith="off", **kw).run()
    assert np.array_equal(auto.results.counts, off.results.counts)
    want = rp.rdf_run(u, u.atoms, n_bins=50, range=(0.0, 2.5))
    assert np.array_equal(auto.results.counts, want["counts"])


def test_every_instance_runs():
    """EXCL x LOWER x AUDIT: the eight instances of rdf_tri_cells_filter_kernel, each
    seen running in the statistics."""
    rng = np.random.default_rng(9)
    h = _cell(_scaled(TO, 14.0))
    r_hi = _width(h) / 3.2
    p = _fluid(2500, h, rng)[None]
    for exclusion in (None, (2, 2)):
        for r_lo in (0.0, 1.0):
            off, _, _ = _run(p, h[None], 30, (r_lo, r_hi), "off", exclusion=exclusion)
            for arith in ("on", "audit"):
                got, st, _ = _run(p, h[None], 30, (r_lo, r_hi), arith, exclusion=exclusion)
                assert np.array_equal(got, off)
                assert st["triclinic_frames"] == 1 and st["audit_violations"] == 0
                assert (st["audit_uncertain_pairs"] > 0) == (arith == "audit")


def test_one_full_frame_audited_at_scale():
    """500,000 particles in a rhombic dodecahedron, rho* = 0.8, range (0, 2.5), audited."""
    rng = np.random.default_rng(10)
    n = 500_000
    unit = _cell(RD).astype(np.float64)
    L = (n / 0.8 / abs(np.linalg.det(unit))) ** (1 / 3)
    h = _cell(_scaled(RD, L))
    p = _fluid(n, h, rng)[None]
    aud, st, ev = _run(p, h[None], 100, (0.0, 2.5), "audit")
    off, _, ev_off = _run(p, h[None], 100, (0.0, 2.5), "off")
    assert np.array_equal(aud, off)
    assert st["audit_violations"] == 0 and st["triclinic_frames"] == 1
    assert st["audit_uncertain_pairs"] > 0 and ev == ev_off
