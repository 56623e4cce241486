"""GPU: the unclamped body of the all-pairs fp32 filter (rdf_filter.cu).

A half-box frame whose every reachable slot is a word of the block histogram adds each
pair at its fp32 slot without a clamp; slots outside the range are scratch words.  Each
case compares exact counts against the fp64 kernel (arith="off") and runs the audit,
which also counts a pair of an unclamped frame that leaves the histogram as a violation,
and checks which frames ran unclamped (`unclamped_frames` of the filter statistics).
The layouts the cases expect follow rdf_filter.cu::filter_plan: the histogram covers the
largest reachable slot of the batch's boxes if that fits two blocks' shared memory at the
clamped layout's column count and costs at most one fraction bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _structure():
    from mdhelper_b200.analysis import structure
    return structure


def _audited(p1, p2, n_bins, rng_, dims, **kw):
    """Counts with arith="audit" (0 violations), equal to arith="off" and "auto"."""
    S = _structure()
    st = {}
    got = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", arith="audit",
                             stats=st, **kw)
    assert st["eligible"] == 1 and st["audit_violations"] == 0, st
    off = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", arith="off", **kw)
    assert np.array_equal(got, off)
    auto = S.radial_histogram(p1, p2, n_bins, rng_, dims, mode="allpairs", **kw)
    assert np.array_equal(auto, off)
    return got, st


def _box(edges):
    return np.array(list(edges) + [90, 90, 90], np.float32)


def test_config2_frame():
    """One frame of the benchmark workload (10k x 10k cation-anion, 201 bins to 14.5):
    its corner distance is slot ~352, above the 203 slots of the clamped layout."""
    from mdhelper_b200 import synthetic
    u, cat, an = synthetic.electrolyte(20_000, 1, seed=20260002)
    S = _structure()
    kw = dict(n_bins=201, range=(0.0, 14.5), mode="allpairs", verbose=False)
    off = S.RadialDistributionFunction(cat, an, arith="off", **kw).run().results.counts
    for arith in ("audit", "auto"):
        r = S.RadialDistributionFunction(cat, an, arith=arith, **kw).run()
        st = r._filter_stats
        assert np.array_equal(r.results.counts, off), arith
        assert st["audit_violations"] == 0
        assert st["halfbox_frames"] == 1 and st["rint_frames"] == 0, st
        assert st["unclamped_frames"] == 1, st
        if arith == "audit":      # one fraction bit fewer: still about 1 pair in 1,000
            assert 0 < st["audit_uncertain_pairs"] < 4e5


def _corner_pairs(box, n, rng, eps):
    """Pairs whose differences sit at h on every axis (the largest minimum-image distance
    ||h||), or at h on some axes and 0 on the others, each moved by a few float32 ulps.
    Both groups stay within [0, box], so the frame takes the half-box form."""
    h = box / 2
    base = (rng.random((n, 3)) * h).astype(np.float32)
    corner = rng.random((n, 3)) < 0.8
    off = np.where(corner, h, 0 * h) + eps * rng.integers(-4, 5, size=(n, 3)) * h
    return base, np.clip(base + off, 0, box).astype(np.float32)


def test_box_corner_and_the_largest_reachable_slot():
    rng = np.random.default_rng(352)
    edges = np.array([11.0, 12.5, 13.25], np.float32)
    dims = _box(edges)
    p1, p2 = _corner_pairs(edges, 3000, rng, 2.0 ** -23)
    # the range ends well below ||h|| (~10.7): the corner pairs land ~100 slots above it
    for n_bins, rng_ in [(120, (0.0, 5.5)), (201, (0.0, 10.5)), (64, (0.0, 10.7))]:
        _, st = _audited(p1, p2, n_bins, rng_, dims, wrap="never")
        assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == 1, st


def test_lower_range_limit_with_pairs_below_it():
    rng = np.random.default_rng(77)
    dims = _box([10.75, 11.5, 12.25])
    p1 = (rng.random((1500, 3)) * dims[:3]).astype(np.float32)
    p2 = (rng.random((2100, 3)) * dims[:3]).astype(np.float32)
    # close pairs: many distances below r_lo, some exactly 0
    p2[:300] = p1[:300] + rng.normal(0, 0.3, (300, 3)).astype(np.float32)
    p2[300:320] = p1[300:320]
    # lo = 50 and 63 scratch slots below bin 0, both unclamped; (100, (1.0, 4.5)) and
    # (37, (2.25, 2.75)) would lose 2 and 4 fraction bits: the clamped layout
    for n_bins, rng_, unclamped in [(200, (1.0, 5.0), 1), (50, (5.0, 9.0), 1),
                                    (100, (1.0, 4.5), 0), (37, (2.25, 2.75), 0)]:
        _, st = _audited(p1, p2, n_bins, rng_, dims)
        assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == unclamped, st


def test_batch_mixing_unclamped_clamped_and_rint_frames():
    """One call whose frames take all three bodies: half-box frames of the ~10-unit boxes
    (unclamped: 305 slots, 150 bins to 4.5), one half-box frame of a 400-unit box, which
    reaches slot ~11,000 and keeps the clamped body, and frames several boxes away (rint
    form)."""
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    rng = np.random.default_rng(5)
    F, n1, n2 = 5, 1300, 1700
    box = np.array([[9.5, 10.25, 11.0], [9.75, 9.5, 10.0], [400.0, 380.0, 390.0],
                    [10.5, 10.5, 10.5], [9.25, 11.5, 10.0]], np.float32)
    spread = np.array([[0.0, 1.0], [-3.0, 4.0], [0.0, 1.0], [0.0, 1.0], [-2.0, 3.0]])
    p1 = np.empty((F, n1, 3), np.float32)
    p2 = np.empty((F, n2, 3), np.float32)
    for f in range(F):
        a, b = spread[f]
        p1[f] = (a + rng.random((n1, 3)) * (b - a)) * box[f]
        p2[f] = (a + rng.random((n2, 3)) * (b - a)) * box[f]
    # the large frame: a dense cluster, so that it has pairs in range
    p2[2, :400] = p1[2, :400] + rng.normal(0, 1.0, (400, 3)).astype(np.float32)
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
        assert st["halfbox_frames"] == 3 and st["rint_frames"] == 2, st
        assert st["unclamped_frames"] == 2, st


@pytest.mark.parametrize("n_bins,edge,unclamped", [(1000, 12.0, 1), (3000, 12.0, 1),
                                                   (3000, 15.0, 0)])
def test_histogram_that_does_not_fit_falls_back(n_bins, edge, unclamped):
    """Bins to 6.0: 1,000 bins in a 12.0 box reach slot ~1,730 (8 columns, as the clamped
    layout), 3,000 bins slot ~5,200 (2 columns, 110 KB: fits); 3,000 bins in a 15.0 box
    reach slot ~6,500, 52 KB more than two blocks' shared memory at 2 columns (falls back
    to the clamped layout)."""
    rng = np.random.default_rng(n_bins)
    dims = _box([edge] * 3)
    p = (rng.random((1200, 3)) * edge).astype(np.float32)
    q, r = _corner_pairs(np.array([edge] * 3, np.float32), 600, rng, 2.0 ** -23)
    _, st = _audited(np.concatenate([p, q]), np.concatenate([p, r]), n_bins, (0.0, 6.0),
                     dims, wrap="never")
    assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == unclamped, st


def test_exclusions():
    rng = np.random.default_rng(78)
    dims = _box([9.5, 9.5, 9.5])
    p = (rng.random((1800, 3)) * dims[:3]).astype(np.float32)
    q = (rng.random((1200, 3)) * dims[:3]).astype(np.float32)
    _, st = _audited(p, p, 120, (0.0, 4.75), dims, exclusion=(3, 3))
    assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == 1, st
    _, st = _audited(p, q, 120, (0.5, 4.75), dims, exclusion=(3, 2))
    assert st["halfbox_frames"] == 1 and st["unclamped_frames"] == 1, st
