"""GPU: the fp32 filter of the triclinic all-pairs path (rdf_tri_filter_kernel) gives the
counts of the restated reference (the CPU oracle of _threshold_pairs) and of the 27-image
kernel (arith "off"), bit for bit; the audit finds no certified pair in a wrong bin."""
import numpy as np
import pytest

from _threshold_pairs import tri_ref_d2, wrap

pytestmark = pytest.mark.gpu

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)              # rhombic dodecahedron
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)          # truncated octahedron
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)           # strongly tilted monoclinic


def _cell(shape, L):
    from oracle import reference_port as rp
    d = np.array([L * shape[0], L * shape[1], L * shape[2], *shape[3:]], np.float32)
    return rp.triclinic_vectors(d).astype(np.float32)


def _fluid(n, h, rng, lo=0.0, hi=1.0):
    return ((rng.random((n, 3)) * (hi - lo) + lo) @ h.astype(np.float64)).astype(np.float32)


def _R(h):
    return 0.5 * float(min(h[0, 0], h[1, 1], h[2, 2]))


def _run(p, cells, n_bins, rng_, arith, *, q=None, exclusion=None, device=False,
         drop_axis=None):
    """One accumulate call, all-pairs path (same group unless q is given)."""
    import torch
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    F, n = p.shape[:2]
    m = n if q is None else q.shape[1]
    ctx = _lib.Context(0)
    try:
        ctx.rdf_set_filter(arith)
        ctx.rdf_configure(n, m, q is None, squared_thresholds(n_bins, rng_), rng_[0], rng_[1],
                          mode="allpairs", exclusion=exclusion, drop_axis=drop_axis)
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
        i, j = np.meshgrid(np.arange(len(a)), np.arange(len(b)), indexing="ij")
        i, j = i.ravel(), j.ravel()
        if exclusion is not None:
            keep = i // exclusion[0] != j // exclusion[1]
            i, j = i[keep], j[keep]
        d2 = tri_ref_d2(a[i], b[j], cells[f])
        k = np.searchsorted(thr, d2, side="right") - 1
        k = k[(k >= 0) & (k < n_bins)]
        out += np.bincount(k, minlength=n_bins)
    return out


def _check(p, cells, n_bins, rng_, *, oracle=True, **kw):
    got, st, ev = _run(p, cells, n_bins, rng_, "auto", **kw)
    off, st_off, ev_off = _run(p, cells, n_bins, rng_, "off", **kw)
    aud, st_aud, _ = _run(p, cells, n_bins, rng_, "audit", **kw)
    assert got.sum() > 0
    assert np.array_equal(got, off), kw
    assert np.array_equal(aud, off), kw
    if oracle:
        want = _oracle(p, cells, n_bins, rng_, q=kw.get("q"), exclusion=kw.get("exclusion"),
                       drop_axis=kw.get("drop_axis"))
        assert np.array_equal(got, want), kw
    assert st_aud["audit_violations"] == 0, st_aud
    assert st_aud["triclinic_frames"] > 0 and st_aud["audit_uncertain_pairs"] >= 0
    assert st["triclinic_frames"] == p.shape[0] and st["declined_frames"] == 0, st
    assert st_off["triclinic_frames"] == 0
    # the filter evaluates the pairs of its tile pairs (same group: the upper triangle)
    F, n = p.shape[:2]
    m = n if kw.get("q") is None else kw["q"].shape[1]
    assert ev_off == F * n * m
    assert (ev <= ev_off) and (ev >= F * n * m // 2)
    return st_aud


@pytest.mark.parametrize("shape,L", [(RD, 20.0), (TO, 22.0), (TILT, 18.0)])
def test_same_group_and_two_groups(shape, L):
    rng = np.random.default_rng(1)
    h = _cell(shape, L)
    cells = np.stack([h, h])
    r_hi = 0.8 * _R(h)
    p = np.stack([_fluid(1500, h, rng), _fluid(1500, h, rng)])
    _check(p, cells, 60, (0.0, r_hi))
    q = np.stack([_fluid(700, h, rng), _fluid(700, h, rng)])
    _check(p, cells, 60, (0.0, r_hi), q=q)


@pytest.mark.parametrize("exclusion", [(3, 3), (2, 5)])
def test_exclusions(exclusion):
    rng = np.random.default_rng(2)
    h = _cell(RD, 20.0)
    p = _fluid(1200, h, rng)[None]
    q = _fluid(3000, h, rng)[None] if exclusion[0] != exclusion[1] else None
    if q is not None:
        q = q[:, :1200 * exclusion[1] // exclusion[0]]
    _check(p, h[None], 50, (0.0, 6.0), exclusion=exclusion, q=q)


def test_lower_edge_and_many_bins():
    rng = np.random.default_rng(3)
    h = _cell(TO, 24.0)
    p = _fluid(1500, h, rng)[None]
    _check(p, h[None], 40, (1.5, 0.8 * _R(h)))
    _check(p, h[None], 1000, (0.0, 0.8 * _R(h)), oracle=False)


@pytest.mark.parametrize("drop_axis", [0, 1, 2])
def test_drop_axis(drop_axis):
    rng = np.random.default_rng(4)
    h = _cell(RD, 20.0)
    p = _fluid(1500, h, rng)[None]
    _check(p, h[None], 40, (0.0, 5.0), drop_axis=drop_axis)


def test_unwrapped_coordinates_host_and_device():
    rng = np.random.default_rng(5)
    h = _cell(TILT, 18.0)
    p = np.stack([_fluid(1500, h, rng, -2.0, 3.0), _fluid(1500, h, rng, -1.0, 1.0)])
    cells = np.stack([h, h])
    _check(p, cells, 40, (0.0, 0.8 * _R(h)))
    _check(p, cells, 40, (0.0, 0.8 * _R(h)), device=True, oracle=False)


def test_mixed_orthorhombic_and_triclinic_trajectory():
    from mdhelper_b200.universe import SyntheticUniverse
    from mdhelper_b200.analysis import structure as S
    from oracle import reference_port as rp
    rng = np.random.default_rng(6)
    n, L = 1500, 20.0
    dims = np.array([[L, L, L, 60, 60, 90], [L, L, L, 90, 90, 90], [L, L, L, 70.53, 109.47,
                                                                      70.53]], np.float32)
    pos = np.stack([_fluid(n, rp.triclinic_vectors(d), rng) for d in dims])
    u = SyntheticUniverse(pos, dims)
    kw = dict(n_bins=50, range=(0.0, 5.0), verbose=False, mode="allpairs")
    auto = S.RadialDistributionFunction(u.atoms, **kw).run()
    off = S.RadialDistributionFunction(u.atoms, arith="off", **kw).run()
    assert np.array_equal(auto.results.counts, off.results.counts)
    want = rp.rdf_run(u, u.atoms, n_bins=50, range=(0.0, 5.0))
    assert np.array_equal(auto.results.counts, want["counts"])


def test_quirk_of_the_27_images_is_reproduced():
    """Truncated octahedron: for some in-range pairs the shortest image is not among the
    reference's 27 (a fold index of 2); the reference then sees them out of range."""
    rng = np.random.default_rng(7)
    h = _cell(TO, 20.0)
    n = 1500
    p = _fluid(n, h, rng)[None]
    r_hi = 0.9 * _R(h)
    # planted pairs: u = (-6.9, 0.3, -0.2) is the shortest image of dx = u + 2a - b + c
    hd = h.astype(np.float64)
    dxq = np.array([-6.9, 0.3, -0.2]) + 2 * hd[0] - hd[1] + hd[2]
    for k in range(10):
        wi = np.array([0.1, 9.5, 0.1]) + 0.05 * rng.random(3)
        p[0, 2 * k] = wi
        p[0, 2 * k + 1] = wi + dxq + 0.05 * rng.random(3)
    w = wrap(p[0], h).astype(np.float64)
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    i, j = i.ravel(), j.ravel()
    ref = tri_ref_d2(p[0][i], p[0][j], h)
    dx = (w[j].astype(np.float32) - w[i].astype(np.float32)).astype(np.float64)
    m = np.array([(a, b, c) for a in range(-2, 3) for b in range(-2, 3) for c in range(-2, 3)])
    true = np.min([((dx + mm @ h.astype(np.float64)) ** 2).sum(1) for mm in m], axis=0)
    quirk = (true < r_hi ** 2) & (ref > true * (1 + 1e-9))
    assert quirk.sum() > 0
    st = _check(p, h[None], 60, (0.0, r_hi))
    assert st["triclinic_frames"] == 1


def test_declined_frames():
    rng = np.random.default_rng(8)
    h = _cell(RD, 16.0)
    R = _R(h)
    p = np.stack([_fluid(1200, h, rng) for _ in range(3)])
    p[1, 7] = [np.nan, 1.0, 1.0]
    p[2, 9] = [3.0e8 * h[0, 0], 1.0, 2.0]         # 2^28 cells away: the wrap decides
    cells = np.stack([h, h, h])
    got, st, ev = _run(p, cells, 40, (0.0, 0.8 * R), "auto")
    off, _, _ = _run(p, cells, 40, (0.0, 0.8 * R), "off")
    assert np.array_equal(got, off)
    # frame 0 filtered, frame 1 (NaN) declined, frame 2 by the extents after the wrap
    from mdhelper_b200 import _lib
    ext = []
    for f in range(3):
        wf = wrap(p[f], h)
        ext.append(np.concatenate([wf.min(0), wf.max(0)]) if f != 1 else
                   np.array([np.nan] * 6, np.float32))
    win = _lib.triclinic_filter_window(40, 0.0, 0.8 * R, cells, np.array(ext, np.float32))
    filtered = sum(w["eligible"] for w in win)
    assert win[0]["eligible"] == 1 and win[1]["eligible"] == 0
    assert st["triclinic_frames"] == filtered and st["declined_frames"] == 3 - filtered
    # r_hi beyond R: every frame declined, counts and pair evaluations as arith "off"
    got, st, ev = _run(p[:1], cells[:1], 40, (0.0, 1.05 * R), "auto")
    off, _, ev_off = _run(p[:1], cells[:1], 40, (0.0, 1.05 * R), "off")
    assert np.array_equal(got, off)
    assert st["declined_frames"] == 1 and st["triclinic_frames"] == 0 and ev == ev_off


def test_every_instance_runs():
    """EXCL x LOWER x AUDIT: the eight instances of rdf_tri_filter_kernel."""
    rng = np.random.default_rng(9)
    h = _cell(TO, 20.0)
    p = _fluid(1100, h, rng)[None]
    for exclusion in (None, (2, 2)):
        for r_lo in (0.0, 1.0):
            got, st, _ = _run(p, h[None], 30, (r_lo, 6.0), "audit", exclusion=exclusion)
            off, _, _ = _run(p, h[None], 30, (r_lo, 6.0), "off", exclusion=exclusion)
            auto, st2, _ = _run(p, h[None], 30, (r_lo, 6.0), "auto", exclusion=exclusion)
            assert np.array_equal(got, off) and np.array_equal(auto, off)
            assert st["audit_violations"] == 0 and st["triclinic_frames"] == 1
            assert st2["triclinic_frames"] == 1


def test_one_full_frame_audited():
    """10^4 x 10^4 two-group frame in a rhombic dodecahedron, audited."""
    rng = np.random.default_rng(10)
    h = _cell(RD, 40.0)
    p = _fluid(10_000, h, rng)[None]
    q = _fluid(10_000, h, rng)[None]
    got, st, ev = _run(p, h[None], 201, (0.0, 11.0), "audit", q=q)
    off, _, _ = _run(p, h[None], 201, (0.0, 11.0), "off", q=q)
    assert np.array_equal(got, off)
    assert st["audit_violations"] == 0 and st["triclinic_frames"] == 1
    assert st["audit_uncertain_pairs"] > 0 and ev == 10_000 * 10_000
