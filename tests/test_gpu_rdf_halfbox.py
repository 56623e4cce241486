"""GPU: the half-box minimum image of the all-pairs fp32 filter (rdf_filter.cu).

Frames whose coordinate differences all lie within 1.5 box lengths take the half-box
form; every case runs with the audit on (each pair the filter calls certain is checked
against the fp64 arithmetic) and must give the counts of the exact kernel."""
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


def test_config2_frame_takes_the_half_box_form():
    """One frame of the benchmark workload (10k x 10k cation-anion, 201 bins to 14.5)."""
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
        if arith == "audit":      # the window stays about one pair in 1,500
            assert 0 < st["audit_uncertain_pairs"] < 2e5


def test_coordinates_over_one_and_a_half_boxes():
    """Coordinates over [-0.25 box, 1.25 box): differences up to 1.5 box, where the
    half-box form needs the larger rounding term."""
    rng = np.random.default_rng(150)
    dims = _box([10.75, 11.5, 12.25])
    lo, hi = -0.25 * dims[:3], 1.25 * dims[:3]
    p1 = (lo + rng.random((1500, 3)) * (hi - lo)).astype(np.float32)
    p2 = (lo + rng.random((2100, 3)) * (hi - lo)).astype(np.float32)
    _, st = _audited(p1, p2, 201, (0.0, 5.0), dims, wrap="never")
    assert st["halfbox_frames"] == 1 and st["rint_frames"] == 0, st


def test_batch_mixing_half_box_and_unwrapped_frames():
    """One call whose frames alternate between wrapped coordinates (half-box form) and
    coordinates several boxes away (rint form): both forms run in the same launch."""
    from mdhelper_b200 import _lib
    from mdhelper_b200.analysis._binning import squared_thresholds
    rng = np.random.default_rng(4)
    F, n1, n2 = 4, 1300, 1700
    box = np.array([[9.5, 10.25, 11.0], [9.75, 9.5, 10.0], [10.5, 10.5, 10.5],
                    [9.25, 11.5, 10.0]], np.float32)
    spread = np.array([[0.0, 1.0], [-3.0, 4.0], [0.0, 1.0], [-2.0, 3.0]])
    p1 = np.empty((F, n1, 3), np.float32)
    p2 = np.empty((F, n2, 3), np.float32)
    for f in range(F):
        a, b = spread[f]
        p1[f] = (a + rng.random((n1, 3)) * (b - a)) * box[f]
        p2[f] = (a + rng.random((n2, 3)) * (b - a)) * box[f]
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
    assert np.array_equal(out["audit"][0], out["off"][0])
    assert np.array_equal(out["auto"][0], out["off"][0])
    for arith in ("audit", "auto"):
        st = out[arith][1]
        assert st["audit_violations"] == 0 and st["declined_frames"] == 0, st
        assert st["halfbox_frames"] == 2 and st["rint_frames"] == 2, st


def test_lower_range_limit_and_non_cubic_box():
    rng = np.random.default_rng(51)
    dims = _box([10.75, 11.5, 12.25])
    p1 = (rng.random((1500, 3)) * dims[:3]).astype(np.float32)
    p2 = (rng.random((2100, 3)) * dims[:3]).astype(np.float32)
    for n_bins, rng_ in [(100, (1.0, 4.5)), (37, (2.25, 2.75))]:
        _, st = _audited(p1, p2, n_bins, rng_, dims)
        assert st["halfbox_frames"] == 1, st


def test_exclusions():
    rng = np.random.default_rng(77)
    dims = _box([9.5, 9.5, 9.5])
    p = (rng.random((1800, 3)) * dims[:3]).astype(np.float32)
    q = (rng.random((1200, 3)) * dims[:3]).astype(np.float32)
    _, st = _audited(p, p, 120, (0.0, 4.75), dims, exclusion=(3, 3))
    assert st["halfbox_frames"] == 1, st
    _, st = _audited(p, q, 120, (0.0, 4.75), dims, exclusion=(3, 2))
    assert st["halfbox_frames"] == 1, st


@pytest.mark.parametrize("n_bins", [1000, 3000])
def test_many_bins(n_bins):
    rng = np.random.default_rng(n_bins)
    dims = _box([12.0, 12.0, 12.0])
    p = (rng.random((1200, 3)) * 12).astype(np.float32)
    _, st = _audited(p, p, n_bins, (0.0, 6.0), dims)
    assert st["halfbox_frames"] == 1, st


def test_lattice_with_every_distance_on_a_bin_edge():
    """Simple-cubic lattice whose neighbour distances sit exactly on bin edges: most pairs
    are uncertain and go through the exact re-evaluation of the half-box form."""
    n, a = 16, 0.5
    g = np.arange(n, dtype=np.float32) * a
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    dims = _box([n * a] * 3)
    from oracle import reference_port as rp
    want = rp.radial_histogram(p, p, 16, (0.0, 4.0), dims)
    got, st = _audited(p, p, 16, (0.0, 4.0), dims)
    assert np.array_equal(got, want)
    assert st["halfbox_frames"] == 1 and st["deferred_entries"] > 0, st
