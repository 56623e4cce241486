"""GPU: x-clean tile pairs of the all-pairs fp32 filter (rdf_filter.cu, rdf_device.cuh::
filter_cleanx_form).

The filter kernel's groups are sorted by x; a tile pair whose x differences all lie
within (-h, h) after one shift S in {0, +L, -L} takes m_x = (xj - S) - xi as one FADD.
Every case compares exact counts with the fp64 kernel (arith="off"), runs the audit (0
violations) and checks how many pairs were evaluated x-clean (`cleanx_pairs`; launches
with exclusions sort their rows but evaluate every tile pair in the dirty form).  The
single-tile cases (at most 1,024 particles per group) fix the tile extents, so the form of
their only tile pair, and with it the clean count, is known: n1 * n2 or 0."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32 = np.float32


def _structure():
    from mdhelper_b200.analysis import structure
    return structure


def _audited(p1, p2, n_bins, rng_, dims, **kw):
    S = _structure()
    st = {}
    got = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", arith="audit",
                             wrap="never", stats=st, **kw)
    assert st["eligible"] == 1 and st["audit_violations"] == 0, st
    off = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", arith="off",
                             wrap="never", **kw)
    assert np.array_equal(got, off)
    st_auto = {}
    auto = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", wrap="never",
                              stats=st_auto, **kw)
    assert np.array_equal(auto, off)
    assert st_auto["cleanx_pairs"] == st["cleanx_pairs"], (st, st_auto)
    assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == 1, st
    return got, st


def _group(rng, n, xs, L):
    """n particles with y, z uniform in [0, L) and x uniform in [x0, x1], plus the listed
    x values exactly (the tile's extremes)."""
    x0, x1, exact = xs
    p = np.empty((n, 3), F32)
    p[:, 1:] = rng.random((n, 2)) * L
    p[:, 0] = x0 + rng.random(n) * (x1 - x0)
    p[:len(exact), 0] = exact
    return p.astype(F32)


L = F32(12.0)
H = F32(6.0)
DELTA = 12.0 / 2 ** 20                      # the margin of filter_cleanx_form
ULP = float(np.spacing(H))


def _below(x, k):
    return float(np.nextafter(F32(x), F32(-np.inf)) if k == 1 else
                 F32(x) - F32(k * np.spacing(F32(x))))


# (name, i-group x (lo, hi, exact values), j-group x, clean)
SINGLE = [
    # S = 0, the interval's upper end 2 delta below h: clean
    ("s0_high_inside", (0.0, 1.0, [0.0]), (0.0, 5.9, [float(H - F32(2 * DELTA))]), True),
    # ... and half a delta below h, a few ulps below it, exactly at h, a few ulps above it
    ("s0_high_margin", (0.0, 1.0, [0.0]), (0.0, 5.9, [float(H - F32(DELTA / 2))]), False),
    ("s0_high_ulps_below", (0.0, 1.0, [0.0]), (0.0, 5.9, [_below(H, 3)]), False),
    ("s0_high_at_h", (0.0, 1.0, [0.0]), (0.0, 5.9, [float(H)]), False),
    ("s0_high_ulps_above", (0.0, 1.0, [0.0]), (0.0, 5.9, [float(H) + 3 * ULP]), False),
    # the lower end at -h + 2 delta (clean) and -h + delta / 2 (dirty)
    ("s0_low_inside", (0.0, 5.9, [float(H - F32(2 * DELTA)), 0.0]), (0.0, 1.0, [0.0, 1.0]),
     True),
    ("s0_low_margin", (0.0, 5.9, [float(H - F32(DELTA / 2)), 0.0]), (0.0, 1.0, [0.0, 1.0]),
     False),
    # S = +L: j-tile in [L/2, L - ulp] (both ends exactly), i-tile just below 0
    ("s_plus_l", (-1.0, -0.1, [-1.0, -0.1]), (6.0, 12.0, [6.0, _below(L, 1)]), True),
    # S = -L: the mirror image
    ("s_minus_l", (6.0, 12.0, [6.0, _below(L, 1)]), (-1.0, -0.1, [-1.0, -0.1]), True),
    # S = +L would need min_j >= L/2: one particle just below it makes the pair dirty
    ("s_plus_l_sterbenz", (-1.0, -0.1, [-1.0, -0.1]), (6.0, 12.0, [_below(6.0, 1)]), False),
    # both groups over the whole box: dirty
    ("dirty_full_box", (0.0, 12.0, []), (0.0, 12.0, []), False),
]


@pytest.mark.parametrize("name,xi,xj,clean", SINGLE, ids=[c[0] for c in SINGLE])
def test_single_tile_pair(name, xi, xj, clean):
    rng = np.random.default_rng([ord(c) for c in name])
    n1, n2 = 1000, 900
    p1 = _group(rng, n1, xi, L)
    p2 = _group(rng, n2, xj, L)
    dims = np.array([L, L, L, 90, 90, 90], F32)
    # bins up to 10 (> h): pairs at |m_x| ~ h are counted
    got, st = _audited(p1, p2, 100, (0.0, 10.0), dims)
    assert got.sum() > 0
    assert st["cleanx_pairs"] == (n1 * n2 if clean else 0), st


def test_shuffled_config2_frame():
    """One frame of the benchmark workload, both groups randomly permuted: the sort does
    not rely on the generator's lattice order, and most pairs are x-clean."""
    from mdhelper_b200 import synthetic
    u, cat, an = synthetic.electrolyte(20_000, 1, seed=20260002)
    rng = np.random.default_rng(7)
    p1 = np.asarray(cat.positions, F32)[rng.permutation(cat.n_atoms)]
    p2 = np.asarray(an.positions, F32)[rng.permutation(an.n_atoms)]
    dims = np.asarray(u.dimensions, F32)
    _, st = _audited(p1, p2, 201, (0.0, 14.5), dims)
    n = len(p1) * len(p2)
    assert 0.6 * n < st["cleanx_pairs"] < n, st


@pytest.mark.parametrize("n", [3000, 9000])
def test_mixed_tiles_exclusions_same_group_and_lower_limit(n):
    """Uniform groups of several tiles: x-sorted, their tile pairs are partly clean (S = 0
    and both shifts) and partly dirty."""
    rng = np.random.default_rng(n)
    edge = F32(9.5)
    dims = np.array([edge, edge, edge, 90, 90, 90], F32)
    p = (rng.random((n, 3)) * edge).astype(F32)
    q = (rng.random((2 * n // 3, 3)) * edge).astype(F32)
    for a, b, rng_, excl in [(p, q, (0.0, 4.75), None), (p, p, (0.0, 4.75), (3, 3)),
                             (p, q, (0.5, 4.75), (3, 2)), (p, p, (1.0, 6.0), None)]:
        _, st = _audited(a, b, 120, rng_, dims, exclusion=excl)
        if excl is None:
            assert 0 < st["cleanx_pairs"] < len(a) * len(b), (rng_, excl, st)
        else:
            # sorted rows (the tags travel with them), every tile pair in the dirty form
            assert st["cleanx_pairs"] == 0, (rng_, excl, st)


def test_batch_mixing_clean_dirty_and_rint_frames():
    """One call: sorted half-box frames with clean tile pairs, a frame whose groups span
    several boxes (rint form, no clean pairs) and the single-tile S = -L layout."""
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    rng = np.random.default_rng(11)
    F, n1, n2 = 4, 2600, 2100
    box = np.array([[10.0, 10.5, 11.0], [9.75, 9.5, 10.0], [10.5, 10.5, 10.5],
                    [12.0, 12.0, 12.0]], F32)
    p1 = np.empty((F, n1, 3), F32)
    p2 = np.empty((F, n2, 3), F32)
    for f in range(F):
        a, b = (-3.0, 4.0) if f == 1 else (0.0, 1.0)
        p1[f] = (a + rng.random((n1, 3)) * (b - a)) * box[f]
        p2[f] = (a + rng.random((n2, 3)) * (b - a)) * box[f]
    p1[3, :, 0] = 6.0 + rng.random(n1) * 5.9
    p2[3, :, 0] = -1.0 + rng.random(n2) * 0.9
    thr = squared_thresholds(150, (0.0, 4.5))
    out = {}
    for arith in ("audit", "off", "auto"):
        ctx = _lib.Context(0)
        try:
            ctx.rdf_set_filter(arith)
            ctx.rdf_set_prewrap("never")
            ctx.rdf_configure(n1, n2, False, thr, 0.0, 4.5, mode="allpairs")
            ctx.rdf_accumulate(p1, 3 * n1, p2, 3 * n2, box, F)
            out[arith] = (ctx.rdf_fetch(), ctx.rdf_filter_stats())
        finally:
            ctx.close()
    assert out["off"][0].sum() > 0
    assert np.array_equal(out["audit"][0], out["off"][0])
    assert np.array_equal(out["auto"][0], out["off"][0])
    for arith in ("audit", "auto"):
        st = out[arith][1]
        assert st["audit_violations"] == 0 and st["declined_frames"] == 0, st
        assert st["halfbox_frames"] == 3 and st["rint_frames"] == 1, st
        # frame 3 alone: every pair (its 3 x 3 tile pairs are all S = -L)
        assert n1 * n2 < st["cleanx_pairs"] < 3 * n1 * n2, st
    assert out["audit"][1]["cleanx_pairs"] == out["auto"][1]["cleanx_pairs"]
