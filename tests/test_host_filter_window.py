"""CPU: the fp32 RDF filter's window against a bit-level model of the kernels' arithmetic.

The layouts and per-frame windows come from the library's own host code
(mdh_rdf_filter_window: rdf_filter_configure, filter_plan, filter_prepare_frame), the per-pair
float32 arithmetic from the numpy model in _filter_model.py, and the exact answer from the
reference's fp64 arithmetic.  Pairs sit at e +- t w for bin edges e and t in [0, 4], w the
frame's window half-width, with differences inside h, at h, near box and near 1.5 box,
unwrapped by many boxes, with y / z components that make the float32 sum of squares round as
far as it can, on boxes whose float32 inverse is far from 1 / box.  Asserted per frame and
body (unclamped half-box, clamped half-box, rint, cell list):
  - a pair the model calls certain lands in its exact slot (certain = fraction bits >= wlim
    or outside the span: such pairs are never re-evaluated);
  - the model's bin coordinate is within mu (the bound without the window's 1.25 margin) of
    the exact one, for distances up to d_max;
  - an unclamped frame never leaves its histogram.
sqrt.approx is taken at both ends of the largest error the filter accepts (2^-22).
"""
import numpy as np
import pytest

import _filter_model as fm
from mdhelper_b200 import _lib
from mdhelper_b200.analysis._binning import squared_thresholds

SQRT_ERR = 2.0 ** -22


def _box_far_from_inverse(lo, hi):
    """The float32 box in [lo, hi) whose float32 inverse is farthest from 1 / box."""
    b = np.unique(np.linspace(lo, hi, 40001).astype(np.float32)).astype(np.float64)
    eps = np.abs(b * (1.0 / b).astype(np.float32).astype(np.float64) - 1.0)
    return float(b[np.argmax(eps)]), float(eps.max())


def _box_near_inverse(lo, hi):
    b = np.unique(np.linspace(lo, hi, 40001).astype(np.float32)).astype(np.float64)
    eps = np.abs(b * (1.0 / b).astype(np.float32).astype(np.float64) - 1.0)
    return float(b[np.argmin(eps)])


def _range_far_scale(n_bins, j, width):
    """A range of n_bins bins starting at bin j (r_lo * scale an integer, so that the offset
    stays a float32 value) whose bin width is near `width` and whose float32 scale rounds by
    almost 2^-24."""
    w = width * (1 + np.arange(-2000, 2000) * 1e-7)
    s = 1.0 / w
    q = np.abs(s.astype(np.float32).astype(np.float64) / s - 1.0)
    w = float(w[np.argmax(q)])
    return j * w, (j + n_bins) * w


B_EPS, EPS_B = _box_far_from_inverse(120.0, 128.0)
B_EXACT = _box_near_inverse(22.9, 23.1)
R_LO_D2, R_HI_D2 = _range_far_scale(400, 22400, 0.0005)

HB = ("inside", "axis", "h", "box", "1.5box", "d2")
# (id, n_bins, r_lo, r_hi, drop_axis, ipt, occ, frames); a frame is (box, form) with form
# "half" (coordinates within 1.5 boxes), "half1" (within one box), "cluster" (a small region
# of a large box: a half-box frame whose reach exceeds the batch's histogram) or "rint"
# (unwrapped by up to 90 % of the eligibility limit)
CASES = [
    ("cfg2-like", 201, 0.0, 14.5, None, 4, 2,
     [((29.24, 29.24, 29.24), "half"), ((400.0, 380.0, 390.0), "cluster"),
      ((29.24, 29.24, 29.24), "rint")]),
    ("corner", 64, 0.0, 10.7, None, 2, 3,
     [((11.0, 12.5, 13.25), "half"), ((11.0, 12.5, 13.25), "rint")]),
    ("one-bin", 1, 0.0, 3.0, None, 4, 4,
     [((7.5, 8.0, 9.0), "half"), ((7.5, 8.0, 9.0), "rint")]),
    ("seven", 7, 0.3, 1.0, None, 2, 2,
     [((2.5, 2.75, 3.0), "half"), ((2.5, 2.75, 3.0), "rint")]),
    ("lower-clamped", 100, 1.0, 4.5, None, 4, 3,
     [((10.75, 11.5, 12.25), "half"), ((10.75, 11.5, 12.25), "rint")]),
    ("lower-shifted", 200, 1.0, 5.0, 1, 4, 2,
     [((10.75, 11.5, 12.25), "half"), ((10.75, 11.5, 12.25), "rint")]),
    ("1000", 1000, 0.0, 6.0, None, 2, 4,
     [((12.0, 12.0, 12.0), "half"), ((12.0, 12.0, 12.0), "rint")]),
    ("4094", 4094, 0.0, 6.0, 2, 4, 2,
     [((12.5, 13.0, 3.0), "half"), ((12.5, 13.0, 3.0), "rint")]),
    ("4095", 4095, 0.5, 6.0, None, 2, 2,
     [((12.0, 12.0, 12.0), "half"), ((12.0, 12.0, 12.0), "rint")]),
    ("4965", 4965, 0.0, 5.0, 0, 4, 2,
     [((3.0, 10.5, 11.0), "half"), ((3.0, 10.5, 11.0), "rint")]),
    ("4965-occ3", 4965, 0.0, 5.0, None, 2, 3,
     [((10.0, 10.5, 11.0), "half1"), ((10.0, 10.5, 11.0), "rint")]),
    # eps_b * D: |box * (float)(1/box) - 1| near 2^-24, differences near one box
    ("eps-b", 1000, 0.0, 5.0, None, 4, 2, [((B_EPS, 20.0, 20.0), "half1")]),
    # (1 + 2^-24)^3 on d2: the scale rounds by almost 2^-24, the inverse box is exact, d2
    # just above 2^7, bins of 1/2000
    ("d2-rounding", 400, R_LO_D2, R_HI_D2, None, 4, 2, [((B_EXACT, 1.0, 1.0), "half1")]),
]


def _ext(lo, hi):
    return np.array([lo] * 3 + [hi] * 3, np.float32)


def _window(case, boxes, exts):
    _, n_bins, r_lo, r_hi, drop, ipt, occ, _ = case
    e1 = np.stack([e[0] for e in exts])
    e2 = np.stack([e[1] for e in exts])
    return _lib.filter_window(n_bins, r_lo, r_hi, boxes, e1, e2, drop_axis=drop, ipt=ipt,
                              filter_occ=occ, sqrt_err=SQRT_ERR)


def _rint_shift(case, box):
    """Boxes of unwrapping at 90 % of the largest the filter accepts for this box."""
    lo, hi = 1, 1 << 21
    while hi - lo > 1:
        mid = (lo + hi) // 2
        ext = _ext(0.0, mid * max(box))
        w = _window(case, np.array([box], np.float32), [(ext, ext)])
        lo, hi = (mid, hi) if w["frames"][0]["allpairs"]["wlim"] > 0 else (lo, mid)
    return max(1, int(0.9 * lo) - 1)


def _region(box, form, r_hi):
    box = np.asarray(box, np.float64)
    if form == "half":
        return 1.5 * box * (1 - 2.0 ** -22)
    if form == "half1":
        return box * (1 - 2.0 ** -22)
    if form == "cluster":
        return np.minimum(box, 3 * r_hi)
    return None


def build_case(case, seed):
    """Frames (box, c, p) of one case, from the edges of its bins."""
    cid, n_bins, r_lo, r_hi, drop, ipt, occ, frames = case
    rng = np.random.default_rng(seed)
    edges = fm.edge_sample(n_bins, r_lo, r_hi, rng)
    out = []
    for box, form in frames:
        box32 = np.array(box, np.float32)
        if form == "rint":
            ns = _rint_shift(case, box)
            region = (ns + 1.0) * box32.astype(np.float64)
            kinds, kw = ("unwrap", "inside"), dict(n_shift=ns)
        else:
            region = _region(box, form, r_hi)
            kinds = ("inside", "axis") if form == "cluster" else HB
            kw = {}
        if drop is not None:
            region = region.copy()
            region[drop] = 1.0
        # the window of the frame's planned extents gives w (the actual extents are within)
        e = _ext(0.0, float(region.max()))
        win = _window(case, box32[None], [(e, e)])
        W, L = win["frames"][0]["allpairs"], win["allpairs"]
        w = fm.window_distance(L, W, n_bins / (r_hi - r_lo)) if W["wlim"] else 1e-6
        c, p = fm.edge_pairs(rng, box32, edges, w, kinds, region, drop=drop, **kw)
        out.append((box32, c, p))
    return out


def run_case(case, seed=1, sqrt_err=SQRT_ERR):
    """Model results per (frame, body) of one case."""
    cid, n_bins, r_lo, r_hi, drop, ipt, occ, frames = case
    fr = build_case(case, seed)
    boxes = np.stack([f[0] for f in fr])
    exts = [fm.extents(c, p) for _, c, p in fr]
    win = _window(case, boxes, exts)
    thr = squared_thresholds(n_bins, (r_lo, r_hi))
    scale = n_bins / (r_hi - r_lo)
    results = []
    for f, (box, c, p) in enumerate(fr):
        Wa, Wc = win["frames"][f]["allpairs"], win["frames"][f]["cells"]
        if Wa["wlim"]:
            body = ("unclamped" if Wa["unclamped"] else "clamped") if Wa["halfbox"] else "rint"
            r = fm.check_pairs(c, p, box, thr, win["allpairs"], Wa,
                               "clamped" if body == "rint" else body, sqrt_err, r_lo, scale,
                               n_bins)
            results.append((cid, f, body, frames[f][1], r, Wa["mu"]))
        if Wc["wlim"]:
            for sb in range(win["clamped"]["sb"] + 1):
                r = fm.check_pairs(c, p, box, thr, win["clamped"], Wc, "cells", sqrt_err, r_lo,
                                   scale, n_bins, sb=sb)
                results.append((cid, f, f"cells-sb{sb}", frames[f][1], r, Wc["mu"]))
    return win, results


_CACHE = {}


def _results(case):
    if case[0] not in _CACHE:
        _CACHE[case[0]] = run_case(case)
    return _CACHE[case[0]]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_certain_pairs_land_in_their_exact_slot(case):
    _, results = _results(case)
    assert results
    for cid, f, body, form, r, mu in results:
        assert r["n"] > 0, (cid, f, body)
        assert r["wrong"] == 0, (cid, f, body, r)
        assert r["outside"] == 0, (cid, f, body, r)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_coordinate_error_within_mu(case):
    _, results = _results(case)
    for cid, f, body, form, r, mu in results:
        assert r["err"] <= mu, (cid, f, body, r["err"], mu)


def test_every_body_runs_and_the_bound_is_probed():
    """Across the cases every body has frames, and the largest observed error reaches at
    least a quarter of mu in each form (else the pairs do not probe the bound)."""
    ratio = {}
    for case in CASES:
        _, results = _results(case)
        for cid, f, body, form, r, mu in results:
            key = "cells" if body.startswith("cells") else body
            ratio[key] = max(ratio.get(key, 0.0), r["err"] / mu)
    print("largest error / mu per body:", {k: round(v, 3) for k, v in ratio.items()})
    assert set(ratio) == {"unclamped", "clamped", "rint", "cells"}, ratio
    for key, v in ratio.items():
        assert v >= 0.25, (key, v)


def test_expected_layouts_and_forms():
    """The cases reach what they are meant to: cfg2's unclamped batch layout (k 13, 353
    slots) with a clamped large-box frame; a LOWER layout; the largest bin counts; the
    probe frames' half-box form."""
    win, res = _results(CASES[0])
    L = win["allpairs"]
    assert (L["k"], L["hslots"], L["unclamped"], L["lo"]) == (13, 353, 1, 0)
    assert win["clamped"]["k"] == 14
    bodies = {(f, b) for _, f, b, *_ in res}
    assert {(0, "unclamped"), (1, "clamped"), (2, "rint")} <= bodies
    win, _ = _results(CASES[4])
    assert win["allpairs"]["lower"] == 1 and win["allpairs"]["unclamped"] == 0
    win, _ = _results(CASES[5])
    assert win["allpairs"]["lower"] == 0 and win["allpairs"]["lo"] == 50
    for i, k in ((8, 9), (9, 9), (10, 9), (7, 10)):
        assert _results(CASES[i])[0]["clamped"]["k"] == k
    for case in CASES[-2:]:
        win, res = _results(case)
        assert win["frames"][0]["allpairs"]["halfbox"] == 1
    assert EPS_B > 0.9 * 2.0 ** -24


def test_declined_frames_and_configurations():
    """Coordinates 2^20 boxes apart, or non-finite ones, leave the frame to the exact kernel;
    8191 bins (k < 9) and a sqrt error above 2^-22 leave the configuration to it."""
    box = np.array([[10.0, 10.0, 10.0]] * 3, np.float32)
    e_ok = _ext(0.0, 10.0)
    e_far = _ext(0.0, 10.0 * 2 ** 20)
    e_nan = e_ok.copy()
    e_nan[4] = np.nan
    w = _lib.filter_window(100, 0.0, 4.0, box, np.stack([e_ok, e_far, e_nan]))
    assert [f["allpairs"]["wlim"] > 0 for f in w["frames"]] == [True, False, False]
    assert [f["cells"]["wlim"] > 0 for f in w["frames"]] == [True, False, False]
    with pytest.raises(ValueError):
        _lib.filter_window(8191, 0.0, 4.0, box[:1], e_ok[None])
    with pytest.raises(ValueError):
        _lib.filter_window(100, 0.0, 4.0, box[:1], e_ok[None], sqrt_err=2.0 ** -21)
    assert _lib.filter_window(4965, 0.0, 4.0, box[:1], e_ok[None])["clamped"]["k"] == 9


def test_model_fma_is_correctly_rounded():
    """fma32 against exact rational arithmetic, ties and near-ties included."""
    from fractions import Fraction
    rng = np.random.default_rng(3)
    a = rng.normal(size=3000).astype(np.float32)
    b = rng.normal(size=3000).astype(np.float32)
    c = (-(a.astype(np.float64) * b) * (1 + rng.normal(size=3000) * 1e-7)).astype(np.float32)
    # exact ties: a * b + c halfway between two floats
    a[:50] = np.float32(1.0) + np.float32(2.0 ** -23)
    b[:50] = np.float32(1.0) + np.float32(2.0 ** -23) * rng.integers(1, 8, 50).astype(np.float32)
    c[:50] = np.float32(-1.0)
    got = fm.fma32(a, b, c)
    for x, y, z, g in zip(a, b, c, got):
        ex = Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z))
        lo = np.float32(float(ex))
        cands = [np.nextafter(lo, np.float32(-np.inf)), lo, np.nextafter(lo, np.float32(np.inf))]
        dist = [abs(Fraction(float(q)) - ex) for q in cands]
        best = min(dist)
        ok = [q for q, dd in zip(cands, dist) if dd == best]
        if len(ok) == 2:                          # tie: even mantissa
            ok = [q for q in ok if not (int(q.view(np.uint32)) & 1)]
        assert g == ok[0], (x, y, z, g, ok)


def test_reference_pinned_against_the_oracle():
    """The exact reference of the model equals the CPU oracle's histogram on a few hundred
    edge pairs, wrapped and unwrapped."""
    from oracle import reference_port as rp
    rng = np.random.default_rng(11)
    box = np.array([10.75, 11.5, 12.25], np.float32)
    n_bins, rr = 40, (0.5, 5.0)
    edges = fm.edge_sample(n_bins, *rr, rng, n_max=12)
    c, p = fm.edge_pairs(rng, box, edges, 1e-6, ("inside", "box", "unwrap"),
                         3 * box.astype(np.float64), n_shift=1)
    c, p = c[:25], p[:300]
    dims = np.array(list(box) + [90, 90, 90], np.float32)
    want = rp.radial_histogram(c, p, n_bins, rr, dims, method="bruteforce")
    df = (p[None, :, :] - c[:, None, :]).reshape(-1, 3)
    slots = fm.ref_slots(fm.ref_d2(df, box), squared_thresholds(n_bins, rr))
    got = np.bincount(slots, minlength=n_bins + 2)[1:n_bins + 1]
    assert want.sum() > 0 and np.array_equal(got, want)
