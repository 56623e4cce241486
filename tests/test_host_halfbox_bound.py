"""CPU: the half-box minimum image of the fp32 filter and its error bound.

The all-pairs filter kernel (csrc/rdf_device.cuh::filter_d2<true>) computes, per axis and
with h = box / 2,
    e = fl(|df| - h)        m = fl(|e| - h)
and filter_prepare_frame bounds ||m| - minimum image of df| by 2^-24 h when every
|df| <= box and by 2^-23 h when every |df| <= 1.5 box; frames with a larger coordinate
difference keep the rint form.  numpy float32 arithmetic rounds to nearest like FADD2,
so these two operations are restated here bit for bit and checked against the exact
minimum image (rational arithmetic).
"""
from fractions import Fraction

import numpy as np
import pytest

E24 = 2.0 ** -24


def halfbox_m(df, box):
    """|m| of the device code, float32 throughout."""
    df = np.asarray(df, dtype=np.float32)
    h = np.float32(box) * np.float32(0.5)
    e = np.abs(df) - h
    return np.abs(np.abs(e) - h)


def exact_min_image(df, box):
    """Distance of df to the nearest multiple of box, exactly."""
    d, b = Fraction(float(df)), Fraction(float(box))
    n = round(d / b)
    return min(abs(d - k * b) for k in (n - 1, n, n + 1))


def axis_bound(D, box):
    """fp32 term of the per-axis bound for a frame whose |df| are all <= D."""
    h = 0.5 * float(box)
    return E24 * (h if D <= float(box) else 2.0 * h)


def halfbox_eligible(lo1, hi1, lo2, hi2, box):
    """The per-axis eligibility rule of filter_prepare_frame (extents in float32)."""
    D = max(float(hi2) - float(lo1), float(hi1) - float(lo2), 0.0) * (1.0 + 2.0 * E24)
    return D <= 1.5 * float(box)


def check(dfs, box):
    dfs = np.asarray(dfs, dtype=np.float32)
    assert np.all(np.isfinite(dfs)) and np.all(np.abs(dfs) <= 1.5 * np.float64(box))
    m = halfbox_m(dfs, box)
    D = float(np.max(np.abs(dfs)))
    bound = Fraction(axis_bound(D, box))
    for df, mf in zip(dfs, m):
        err = abs(Fraction(float(mf)) - exact_min_image(df, box))
        # per pair: the bound of the narrowest frame containing this |df|
        assert err <= Fraction(axis_bound(abs(float(df)), box)), (float(df), float(box))
        assert err <= bound


BOXES = [np.float32(29.24), np.float32(10.0), np.float32(1.0), np.float32(3.3333333),
         np.float32(1234.5678), np.float32(0.0071)]


@pytest.mark.parametrize("box", BOXES, ids=lambda b: f"{float(b):g}")
def test_random_differences(box):
    rng = np.random.default_rng(int(float(box) * 1000) % 2**32)
    b = float(box)
    for lim in (0.5 * b, b, 1.5 * b):
        df = (rng.uniform(-lim, lim, 4000)).astype(np.float32)
        df = df[np.abs(df.astype(np.float64)) <= 1.5 * b]
        check(df, box)


def _ulps_around(x, k=4):
    x = np.float32(x)
    out = [x]
    up = dn = x
    for _ in range(k):
        up = np.nextafter(up, np.float32(np.inf))
        dn = np.nextafter(dn, np.float32(-np.inf))
        out += [up, dn]
    return out


@pytest.mark.parametrize("box", BOXES, ids=lambda b: f"{float(b):g}")
def test_adversarial_differences(box):
    b = np.float32(box)
    h = b * np.float32(0.5)
    centres = [np.float32(0.0), np.float32(1e-45), np.float32(1e-39), np.float32(1.17e-38),
               h * np.float32(0.5), h, b, np.float32(1.5) * b, h * np.float32(1.5),
               np.float32(1e-7) * b]
    vals = []
    for c in centres:
        for v in _ulps_around(c):
            vals += [v, -v]
    vals = np.array(vals, dtype=np.float32)
    vals = vals[np.abs(vals.astype(np.float64)) <= 1.5 * float(b)]
    check(vals, b)


def test_non_cubic_box_axes_use_their_own_bound():
    """Each axis is bounded with its own box length (a 3:1:0.1 box)."""
    rng = np.random.default_rng(7)
    for box in (np.float32(30.0), np.float32(10.0), np.float32(1.0)):
        df = rng.uniform(-1.5 * float(box), 1.5 * float(box), 3000).astype(np.float32)
        df = df[np.abs(df.astype(np.float64)) <= 1.5 * float(box)]
        check(df, box)


def test_differences_above_one_box_need_the_larger_term():
    """Some |df| > box rounds by more than 2^-24 h: the bound of such frames cannot be
    the one of frames within one box."""
    rng = np.random.default_rng(11)
    box = np.float32(29.24)
    df = rng.uniform(float(box), 1.5 * float(box), 20000).astype(np.float32)
    m = halfbox_m(df, box)
    worst = max(abs(Fraction(float(x)) - exact_min_image(d, box)) for d, x in zip(df, m))
    assert worst > Fraction(E24 * 0.5 * float(box))


def test_eligibility_rule():
    box = np.float32(29.24)
    b = float(box)
    # coordinates spread over [-0.25 box, 1.25 box): the largest difference is 1.5 box
    # minus a little -- eligible only if the rounding margin still fits
    lo = np.float32(-0.25 * b)
    hi = np.nextafter(np.float32(1.25 * b), np.float32(-np.inf))
    assert halfbox_eligible(np.float32(0), box * np.float32(0.999), np.float32(0),
                            box * np.float32(0.999), box)
    assert halfbox_eligible(np.float32(0), np.float32(1.4 * b), np.float32(0),
                            np.float32(1.4 * b), box)
    # D_k > 1.5 box_k is rejected, also by one ulp, and unwrapped frames are
    assert not halfbox_eligible(np.float32(0), np.float32(1.5) * box, np.float32(0),
                                np.float32(1.5) * box, box)
    assert not halfbox_eligible(np.float32(0), np.float32(1.6 * b), np.float32(0),
                                np.float32(1.6 * b), box)
    assert not halfbox_eligible(np.float32(-3 * b), np.float32(4 * b), np.float32(-3 * b),
                                np.float32(4 * b), box)
    # the rule uses both cross differences of the two groups
    assert not halfbox_eligible(np.float32(0), np.float32(0.1 * b), np.float32(1.55 * b),
                                np.float32(1.56 * b), box)
    # what an accepted frame guarantees: every float32 difference within 1.5 box
    if halfbox_eligible(lo, hi, lo, hi, box):
        assert float(np.float32(hi - lo)) <= 1.5 * b
    # and why the rule exists: past 1.5 box the half-box form is no minimum image
    df = np.float32(1.6 * b)
    assert abs(Fraction(float(halfbox_m(df, box))) - exact_min_image(df, box)) > b / 10
