"""CPU: the x-clean form of the all-pairs fp32 filter, restated in float32 (rdf_device.cuh::
filter_cleanx_form, filter_d2<HALF, CX>; DESIGN.md section 4.1b).

A tile pair is x-clean with shift S when every x difference xj - xi of its tiles lies in
(-h + delta, h - delta) after subtracting S (h = L/2, delta = 2^-20 L).  Then m_x is one
rounded float32 addition of the shifted operands -- xj - L (S = +L) and L - xi (S = -L)
are exact by Sterbenz -- and, against the exact minimum image of the reference's float32
difference df = fl(xj - xi), it errs by at most 2^-24 (h + D) with D >= |xj - xi| (the
term filter_prepare_frame adds to the half-box bound on x).  Checked here with exact
rationals at the interval ends (+-h +- a few ulps, the margin), at x = L/2 and L - ulp,
for both shifts, and for dirty tile pairs."""
from fractions import Fraction

import numpy as np
import pytest

F32 = np.float32
E24 = Fraction(1, 2 ** 24)


def cleanx_form(lo_i, hi_i, lo_j, hi_j, L):
    """filter_cleanx_form, in fp64 as the device evaluates it."""
    l = float(L)
    h, dl = 0.5 * l, l / 1048576.0
    lo, hi = float(lo_j) - float(hi_i), float(hi_j) - float(lo_i)
    sj = float(lo_j) >= h and float(hi_j) <= 2.0 * l
    si = float(lo_i) >= h and float(hi_i) <= 2.0 * l
    if lo > -h + dl and hi < h - dl:
        return 1
    if sj and lo - l > -h + dl and hi - l < h - dl:
        return 2
    if si and lo + l > -h + dl and hi + l < h - dl:
        return 3
    return 0


def clean_mx(xi, xj, L, form):
    """The kernel's m_x of an x-clean tile pair: bx + ax with bx = xj (- L for S = +L) and
    ax = -xi (+ L for S = -L), every operation a float32 rounding."""
    bx = F32(xj) - F32(L) if form == 2 else F32(xj)
    ax = -F32(xi) + F32(L) if form == 3 else -F32(xi)
    return F32(bx + ax), F32(bx), F32(ax)


def exact_min_image(df, L):
    """|df - L round(df / L)| exactly (ties: either image, the same magnitude)."""
    q = Fraction(float(df)) / Fraction(float(L))
    n = (q.numerator * 2 + q.denominator) // (2 * q.denominator)
    return abs(Fraction(float(df)) - n * Fraction(float(L)))


def check_tiles(xi, xj, L):
    """Classifies the tile pair and, if clean, checks every pair: the shifts are exact and
    | |m_x| - min_image(df) | <= 2^-24 (h + D).  Returns the form."""
    xi, xj = np.asarray(xi, F32), np.asarray(xj, F32)
    form = cleanx_form(xi.min(), xi.max(), xj.min(), xj.max(), L)
    if form == 0:
        return 0
    Lf = Fraction(float(L))
    S = {1: 0, 2: Lf, 3: -Lf}[form]
    h = Lf / 2
    D = max(Fraction(float(xj.max())) - Fraction(float(xi.min())),
            Fraction(float(xi.max())) - Fraction(float(xj.min())))
    bound = E24 * (h + D)
    worst = Fraction(0)
    for a in xi:
        for b in xj:
            m, bx, ax = clean_mx(a, b, L, form)
            # the shifted operands are exact
            assert Fraction(float(bx)) == Fraction(float(b)) - (S if form == 2 else 0)
            assert Fraction(float(ax)) == -Fraction(float(a)) + (Lf if form == 3 else 0)
            v = Fraction(float(b)) - Fraction(float(a)) - S
            assert abs(v) < h
            df = F32(F32(b) - F32(a))
            err = abs(abs(Fraction(float(m))) - exact_min_image(df, L))
            assert err <= bound, (float(a), float(b), form, float(err), float(bound))
            worst = max(worst, err)
    return form


L = F32(12.0)
H = 6.0
DELTA = 12.0 / 2 ** 20


def _up(x, k):
    x = F32(x)
    for _ in range(k):
        x = np.nextafter(x, F32(np.inf))
    return x


def _down(x, k):
    x = F32(x)
    for _ in range(k):
        x = np.nextafter(x, F32(-np.inf))
    return x


def _tile(rng, lo, hi, n=40, exact=()):
    t = (F32(lo) + rng.random(n) * (F32(hi) - F32(lo))).astype(F32)
    t[:len(exact)] = exact
    return t


@pytest.mark.parametrize("end,form", [
    (F32(H - 2 * DELTA), 1),            # 2 delta inside: clean
    (F32(H - DELTA / 2), 0),            # inside the margin: dirty
    (_down(H, 3), 0), (F32(H), 0), (_up(H, 3), 0),     # +-h +- a few ulps: dirty
])
def test_interval_end_at_plus_h(end, form):
    rng = np.random.default_rng(1)
    xi = _tile(rng, 0.0, 1.0, exact=[0.0])
    xj = _tile(rng, 0.0, 5.0, exact=[end])
    assert check_tiles(xi, xj, L) == form


@pytest.mark.parametrize("end,form", [
    (F32(H - 2 * DELTA), 1), (F32(H - DELTA / 2), 0), (_down(H, 2), 0), (F32(H), 0),
])
def test_interval_end_at_minus_h(end, form):
    rng = np.random.default_rng(2)
    xi = _tile(rng, 0.0, 5.0, exact=[end, 0.0])
    xj = _tile(rng, 0.0, 1.0, exact=[0.0, 1.0])
    assert check_tiles(xi, xj, L) == form


def test_shift_plus_l_at_half_box_and_below_the_edge():
    """S = +L with the j-tile from exactly L/2 to L - ulp: xj - L is exact at both ends."""
    rng = np.random.default_rng(3)
    xi = _tile(rng, -1.0, -0.1, exact=[-1.0, -0.1])
    xj = _tile(rng, 6.0, 12.0, exact=[F32(6.0), _down(12.0, 1)])
    assert check_tiles(xi, xj, L) == 2
    # one particle one ulp below L/2: Sterbenz no longer covers xj - L, dirty
    xj[2] = _down(6.0, 1)
    assert check_tiles(xi, xj, L) == 0


def test_shift_minus_l_at_half_box_and_below_the_edge():
    rng = np.random.default_rng(4)
    xi = _tile(rng, 6.0, 12.0, exact=[F32(6.0), _down(12.0, 1)])
    xj = _tile(rng, -1.0, -0.1, exact=[-1.0, -0.1])
    assert check_tiles(xi, xj, L) == 3
    # the restore of the negated i-coordinates, (L - xi) - L, gives -xi back exactly
    for a in xi:
        assert F32(F32(-a + L) - L) == -a
    xi[2] = _down(6.0, 1)
    assert check_tiles(xi, xj, L) == 0


def test_shifted_intervals_near_plus_minus_h():
    """S = +L whose shifted interval ends 2 delta inside -h (clean) or inside the margin."""
    rng = np.random.default_rng(5)
    xi = _tile(rng, 0.0, 0.5, exact=[0.0, 0.5])
    for lo_j, form in [(F32(0.5 + H + 2 * DELTA), 2), (F32(0.5 + H + DELTA / 2), 0)]:
        xj = _tile(rng, float(lo_j), 11.0, exact=[lo_j, F32(11.0)])
        assert check_tiles(xi, xj, L) == form


def test_dirty_tile_pairs_need_the_fold():
    """A dirty tile pair whose interval crosses h: the unfolded difference is not the
    minimum image, which is why such pairs keep the half-box form."""
    rng = np.random.default_rng(6)
    xi = _tile(rng, 0.0, 1.0, exact=[0.0])
    xj = _tile(rng, 5.0, 8.0, exact=[F32(8.0)])
    assert check_tiles(xi, xj, L) == 0
    m, _, _ = clean_mx(F32(0.0), F32(8.0), L, 1)
    assert abs(Fraction(float(m))) != exact_min_image(F32(8.0), L)


def test_random_tiles_of_a_sorted_group():
    """Uniform particles sorted by x, 1,024-row tiles of a 20,000-particle frame scaled to
    a few dozen rows: every tile pair the rule calls clean passes the check, and most are
    clean."""
    rng = np.random.default_rng(7)
    Lb = F32(29.24)
    x1 = np.sort(rng.random(400) * Lb).astype(F32)
    x2 = np.sort(rng.random(400) * Lb).astype(F32)
    t1, t2 = np.array_split(x1, 10), np.array_split(x2, 10)
    forms = [check_tiles(a, b, Lb) for a in t1 for b in t2]
    assert forms.count(2) > 0 and forms.count(3) > 0
    assert sum(f != 0 for f in forms) >= 0.6 * len(forms)
