"""GPU: the exact RDF bin lookup of rdf_device.cuh.

1. Audit sweep: the branch-free guess (slot_fast) is checked against the binary search
   (slot_search) for every double d2 >= 0, inf and NaN (mdh_rdf_bin_guess_audit) on the
   configurations of _threshold_pairs.SWEEP: r_lo = 0, and (r - 1, r) from r = 50 to 1000 at
   100 to 4965 bins, on both sides of the host error bound.  A configuration the run uses
   the guess for must have no disagreement; one with disagreements must have been rejected
   by the configure-time self-check.
2. Instance matrix: every instance of the exact pair kernels (all pairs, cell list,
   triclinic all pairs and cell list), FAST and not, on pairs that straddle the thresholds
   (_threshold_pairs.straddle_pairs) plus random fill, one group and two, with and without
   exclusions: counts bit-exact against the CPU oracle.
3. The production fallback: a configuration the self-check rejects runs through the analysis
   class, all pairs and cell list, with the oracle's counts.
4. The lane-private histogram's bin-count edge: 742 bins run, 743 are refused.
"""
import os
import time

import numpy as np
import pytest

import _threshold_pairs as tp

pytestmark = pytest.mark.gpu


def _lib():
    from mdhelper_b200 import _lib
    return _lib


def _thr(n_bins, rr):
    from mdhelper_b200.analysis._binning import squared_thresholds
    return squared_thresholds(n_bins, rr)


class _Tune:
    """MDH_TUNE for the contexts created inside the block."""

    def __init__(self, tune):
        self.tune = tune

    def __enter__(self):
        self.old = os.environ.get("MDH_TUNE")
        os.environ["MDH_TUNE"] = self.tune

    def __exit__(self, *a):
        if self.old is None:
            os.environ.pop("MDH_TUNE", None)
        else:
            os.environ["MDH_TUNE"] = self.old


# ---- 1. audit sweep ------------------------------------------------------------------------

_AUDIT = {}


def _audit(r_lo, r_hi, n_bins):
    key = (r_lo, r_hi, n_bins)
    if key not in _AUDIT:
        ctx = _lib().Context(0)
        try:
            ctx.rdf_configure(10, 10, True, _thr(n_bins, (r_lo, r_hi)), r_lo, r_hi,
                              mode="allpairs")
            look = ctx.rdf_bin_lookup()
            t0 = time.perf_counter()
            au = ctx.rdf_bin_guess_audit()
            ms = 1e3 * (time.perf_counter() - t0)
        finally:
            ctx.close()
        up, down, margin = tp.guess_error_bound(n_bins, r_lo, r_hi)
        print(f"\naudit ({r_lo:g}, {r_hi:g}) {n_bins} bins: fast={look['fast']} "
              f"selfcheck_bad={look['selfcheck_bad']} audit_bad={au['bad']} "
              f"first_bits={au['first_bits']:#x} slot_diff={au['slot_diff']} "
              f"bound={up:.4f} margin={margin:.4f} time={ms:.1f} ms")
        _AUDIT[key] = look, au
    return _AUDIT[key]


@pytest.mark.parametrize("cfg", tp.SWEEP, ids=[f"{a:g}-{b:g}-{n}" for a, b, n in tp.SWEEP])
def test_audit_sweep(cfg):
    r_lo, r_hi, n_bins = cfg
    look, au = _audit(r_lo, r_hi, n_bins)
    assert au["classes"] == tp.N_CLASSES
    where = (cfg, look, au)
    if look["fast"]:
        assert au["bad"] == 0, where
    if au["bad"]:
        assert look["fast"] == 0 and look["selfcheck_bad"] > 0, where
        assert au["slot_diff"] != 0 and au["first_bits"] >= 0, where
    up, down, margin = tp.guess_error_bound(n_bins, r_lo, r_hi)
    if up < margin and down < 1 - margin:
        # the host bound proves the guess for this configuration
        assert au["bad"] == 0 and look["fast"] == 1, where


# ---- 2. instance matrix ------------------------------------------------------------------

def _rp():
    from oracle import reference_port as rp
    return rp


def _cell(dims):
    return _rp().triclinic_vectors(np.asarray(dims, np.float32)).astype(np.float32)


def _groups(box, n_bins, rr, seed, n_fill=600, grid=None, drop=None):
    """Group 1: the centres of the straddling pairs, group 2 their partners, each followed
    by n_fill random particles in the cell; the pair (c_i, p_i) is row i of both."""
    rng = np.random.default_rng(seed)
    thr = _thr(n_bins, rr)
    ks = tp.threshold_sample(n_bins, rng)
    c, p, *_ = tp.straddle_pairs(box, thr, ks, rng, grid=grid, drop=drop)
    h = np.asarray(box, np.float64)
    h = h if h.ndim == 2 else np.diag(h)
    fill = lambda: (rng.random((n_fill, 3)) @ h).astype(np.float32)
    g1, g2 = np.concatenate([c, fill()]), np.concatenate([p, fill()])
    if drop is not None:
        g1[:, drop] = g2[:, drop] = 0
    return g1, g2


def _dims(box):
    box = np.asarray(box, np.float32)
    if box.ndim == 2:
        raise ValueError("pass dims for triclinic cells")
    return np.concatenate([box, [90, 90, 90]]).astype(np.float32)


def _oracle(g1, g2, dims, n_bins, rr, same, excl):
    """Same group: both groups as one (the straddling pairs are pairs within it)."""
    if same:
        g = np.concatenate([g1, g2])
        return _rp().radial_histogram(g, g, n_bins, rr, dims, exclusion=excl,
                                      method="bruteforce")
    return _rp().radial_histogram(g1, g2, n_bins, rr, dims, exclusion=excl, method="bruteforce")


def _run(tune, g1, g2, box, n_bins, rr, same, excl, *, mode, hist="auto", arith="off",
         frames=None):
    """One accumulate call through the C ABI; box [3] edges or a 3x3 cell.  frames: extra
    (g1, g2) frames after the first, same box.  Returns (counts, filter stats, lookup)."""
    L = _lib()
    if same:
        g1, g2 = np.concatenate([g1, g2]), None
        frames = [np.concatenate(f) for f in frames] if frames else None
    a = np.stack([g1] + [f if same else f[0] for f in (frames or [])])
    b = None if same else np.stack([g2] + [f[1] for f in (frames or [])])
    F = len(a)
    with _Tune(tune):                       # read by rdf_configure
        return _run_ctx(L, a, b, F, box, n_bins, rr, same, excl, mode, hist, arith)


def _run_ctx(L, a, b, F, box, n_bins, rr, same, excl, mode, hist, arith):
    ctx = L.Context(0)
    try:
        ctx.rdf_set_filter(arith)
        ctx.rdf_set_prewrap("never")
        n1, n2 = a.shape[1], (a if same else b).shape[1]
        ctx.rdf_configure(n1, n2, same, _thr(n_bins, rr), rr[0], rr[1], exclusion=excl,
                          mode=mode, hist=hist)
        box = np.asarray(box, np.float32)
        if box.ndim == 2:
            ctx.rdf_accumulate_triclinic(a, 3 * n1, b, 3 * n2, np.stack([box] * F), F)
        else:
            ctx.rdf_accumulate(a, 3 * n1, b, 3 * n2, np.stack([box] * F), F)
        return ctx.rdf_fetch(), ctx.rdf_filter_stats(), ctx.rdf_bin_lookup()
    finally:
        ctx.close()


# (box, n_bins, range, grid): a power-of-two box with dyadic edges (d2 == T[k] exactly, and
# inv exact), and r_lo > 0 (T[0]) in an uneven box; both have cells of the cell list
ORTHO = [((32.0, 32.0, 32.0), 64, (0.0, 8.0), 2.0 ** -8),
         ((11.0, 12.5, 13.25), 100, (1.0, 3.5), None)]
SAME_EXCL = [(False, None), (False, (3, 5)), (True, None), (True, (3, 3))]
_DATA, _WANT = {}, {}


def _data(ci):
    if ci not in _DATA:
        box, n_bins, rr, grid = ORTHO[ci]
        _DATA[ci] = _groups(box, n_bins, rr, seed=10 + ci, grid=grid)
    return _DATA[ci]


def _want(ci, same, excl):
    key = (ci, same, excl)
    if key not in _WANT:
        box, n_bins, rr, _ = ORTHO[ci]
        g1, g2 = _data(ci)
        _WANT[key] = _oracle(g1, g2, _dims(box), n_bins, rr, same, excl)
    return _WANT[key]


def _check(got, want, look, fast, where):
    assert want.sum() > 0, where
    assert look["fast"] == fast, (where, look)
    assert np.array_equal(got, want), (where, np.flatnonzero(got != want)[:10],
                                       (got - want)[got != want][:10])


@pytest.mark.parametrize("hist", ["warp_atomic", "lane_private"])
@pytest.mark.parametrize("tune", ["ipt=4", "ipt=2", "ipt=4,fast=0", "ipt=2,fast=0"])
def test_allpairs_instances(hist, tune):
    """rdf_allpairs_kernel<HIST, EXCL, FAST, IPT>: all 16 instances (arith off: the exact
    kernel takes every frame)."""
    fast = 0 if "fast=0" in tune else 1
    for ci, (box, n_bins, rr, _) in enumerate(ORTHO):
        g1, g2 = _data(ci)
        for same, excl in SAME_EXCL:
            got, _, look = _run(tune, g1, g2, box, n_bins, rr, same, excl,
                                      mode="allpairs", hist=hist)
            _check(got, _want(ci, same, excl), look, fast, (hist, tune, ci, same, excl))


@pytest.mark.parametrize("hist", ["warp_atomic", "lane_private"])
@pytest.mark.parametrize("tune", ["", "fast=0"])
def test_cells_instances(hist, tune):
    """rdf_cells_kernel<HIST, EXCL, FAST>: all 8 instances (arith off)."""
    fast = 0 if tune else 1
    for ci, (box, n_bins, rr, _) in enumerate(ORTHO):
        g1, g2 = _data(ci)
        for same, excl in SAME_EXCL:
            got, _, look = _run(tune, g1, g2, box, n_bins, rr, same, excl,
                                      mode="cells", hist=hist)
            _check(got, _want(ci, same, excl), look, fast, (hist, tune, ci, same, excl))


@pytest.mark.parametrize("arith", ["audit", "auto"])
def test_cells_filter_fix_with_binary_search(arith):
    """The cell-pair filter kernel's fp64 re-evaluation (cp_fix) with slot_search."""
    for ci, (box, n_bins, rr, _) in enumerate(ORTHO):
        g1, g2 = _data(ci)
        for same, excl in SAME_EXCL:
            got, st, look = _run("fast=0", g1, g2, box, n_bins, rr, same, excl,
                                       mode="cells", arith=arith)
            where = (arith, ci, same, excl, st)
            _check(got, _want(ci, same, excl), look, 0, where)
            assert st["eligible"] == 1 and st["declined_frames"] == 0, where
            assert st["deferred_entries"] > 0 and st["audit_violations"] == 0, where


RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)
TRI = {"RD": (RD, (0.0, 4.0), 40), "TO": (TO, (0.5, 4.0), 40), "TILT": (TILT, (0.0, 3.5), 35)}


def _tri_case(name):
    shape, rr, n_bins = TRI[name]
    dims = np.array([20 * shape[0], 20 * shape[1], 20 * shape[2], *shape[3:]], np.float32)
    h = _cell(dims)
    g1, g2 = _groups(h, n_bins, rr, seed=list(TRI).index(name) + 30)
    return dims, h, n_bins, rr, g1, g2


@pytest.mark.parametrize("name", list(TRI))
def test_triclinic_instances(name):
    """rdf_triclinic_kernel<EXCL> (all pairs) and rdf_tri_cells_kernel<EXCL, FAST> (cell
    list), RD / TO / TILT cells; a second frame with a particle far outside the cell sends
    the cell-list kernel down its 27-image path (P.far) -- its counts must equal the
    all-pairs kernel's, which the first frame checks against the oracle."""
    dims, h, n_bins, rr, g1, g2 = _tri_case(name)
    far1, far2 = g1.copy(), g2.copy()
    far1[-1] = [1.0e20, -3.0e19, 5.0e19]
    for same, excl in SAME_EXCL:
        want = _oracle(g1, g2, dims, n_bins, rr, same, excl)
        got, _, look = _run("", g1, g2, h, n_bins, rr, same, excl, mode="allpairs")
        _check(got, want, look, 1, (name, "allpairs", same, excl))
        ref2, _, _ = _run("", g1, g2, h, n_bins, rr, same, excl, mode="allpairs",
                          frames=[(far1, far2)])
        for tune, fast in (("", 1), ("fast=0", 0)):
            got, _, look = _run(tune, g1, g2, h, n_bins, rr, same, excl, mode="cells")
            _check(got, want, look, fast, (name, "cells", tune, same, excl))
            got, _, look = _run(tune, g1, g2, h, n_bins, rr, same, excl, mode="cells",
                                      frames=[(far1, far2)])
            _check(got, ref2, look, fast, (name, "cells far", tune, same, excl))


@pytest.mark.parametrize("tune", ["", "fast=0"])
def test_triclinic_flat_grid(tune):
    """drop_axis = 2 on a triclinic cell: the flat cell-list grid, both lookups, through the
    analysis class against the reference's frame loop."""
    from mdhelper_b200.analysis.structure import RadialDistributionFunction
    from mdhelper_b200.universe import SyntheticUniverse
    shape, rr, n_bins = TRI["TILT"]
    dims = np.array([20 * shape[0], 20 * shape[1], 20 * shape[2], *shape[3:]], np.float32)
    flat = dims.copy()
    flat[2] = flat[:3].max()
    g1, g2 = _groups(_cell(flat), n_bins, rr, seed=77, drop=2)
    u = SyntheticUniverse(np.concatenate([g1, g2])[None], dims)
    a, b = u.select(slice(0, len(g1))), u.select(slice(len(g1), len(g1) + len(g2)))
    want = _rp().rdf_run(u, a, b, n_bins=n_bins, range=rr, drop_axis=2)["counts"]
    assert want.sum() > 0
    with _Tune(tune):
        r = RadialDistributionFunction(a, b, n_bins=n_bins, range=rr, drop_axis=2,
                                       mode="cells", verbose=False).run()
    assert np.array_equal(r.results.counts, want)


# ---- 3. production fallback ----------------------------------------------------------------

FALLBACK = [(299.0, 300.0, 1000), (499.0, 500.0, 1000), (999.0, 1000.0, 2000)]


def test_production_fallback():
    """The first configuration of FALLBACK the self-check rejects here, with no MDH_TUNE:
    the analysis class, all pairs and cell list, gives the oracle's counts."""
    from mdhelper_b200.analysis.structure import RadialDistributionFunction
    from mdhelper_b200.universe import SyntheticUniverse
    assert os.environ.get("MDH_TUNE") in (None, "")
    cfg = next((c for c in FALLBACK if _audit(*c)[0]["fast"] == 0), None)
    assert cfg is not None, [_audit(*c) for c in FALLBACK]
    r_lo, r_hi, n_bins = cfg
    box = np.full(3, 3.2 * r_hi, np.float32)
    g1, g2 = _groups(box, n_bins, (r_lo, r_hi), seed=5, n_fill=300)
    u = SyntheticUniverse(np.concatenate([g1, g2])[None], np.concatenate([box, [90] * 3]))
    a, b = u.select(slice(0, len(g1))), u.select(slice(len(g1), len(g1) + len(g2)))
    want = _rp().rdf_run(u, a, b, n_bins=n_bins, range=(r_lo, r_hi))["counts"]
    assert want.sum() > 0
    for mode in ("allpairs", "cells"):
        r = RadialDistributionFunction(a, b, n_bins=n_bins, range=(r_lo, r_hi), mode=mode,
                                       verbose=False).run()
        assert np.array_equal(r.results.counts, want), (cfg, mode)


# ---- 4. lane-private bin-count edge ------------------------------------------------------

@pytest.mark.parametrize("tune", ["ipt=4", "ipt=2"])
def test_lane_private_742_bins(tune):
    """742 bins, the most the lane-private histogram takes (pair_smem_bytes<LANE_PRIVATE, 4>
    <= 227 KB), exact with both tile widths and both lookups."""
    box, rr, n_bins = (11.0, 12.5, 13.25), (0.0, 5.0), 742
    g1, g2 = _groups(box, n_bins, rr, seed=742)
    for t, fast in ((tune, 1), (tune + ",fast=0", 0)):
        for same, excl in [(False, None), (True, (3, 3))]:
            want = _oracle(g1, g2, _dims(box), n_bins, rr, same, excl)
            got, _, look = _run(t, g1, g2, box, n_bins, rr, same, excl,
                                      mode="allpairs", hist="lane_private")
            _check(got, want, look, fast, (t, same, excl))


def test_lane_private_743_bins_are_refused():
    ctx = _lib().Context(0)
    try:
        with pytest.raises(ValueError, match="shared memory"):
            ctx.rdf_configure(10, 10, True, _thr(743, (0.0, 5.0)), 0.0, 5.0,
                              hist="lane_private")
        ctx.rdf_configure(10, 10, True, _thr(742, (0.0, 5.0)), 0.0, 5.0, hist="lane_private")
    finally:
        ctx.close()
