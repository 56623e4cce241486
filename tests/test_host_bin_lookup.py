"""CPU: the pieces the exact bin lookup and its GPU tests rest on.

- _threshold_pairs.straddle_pairs gives pairs on both sides of each threshold T[k], one
  float32 step apart, in the slots the CPU oracle (reference_port.capped_distance +
  numpy.histogram) gives them, with the oracle's distance bit for bit -- orthorhombic,
  triclinic, across periodic faces, T[0] with r_lo > 0 and T[n_bins]; in a power-of-two box
  with dyadic edges d2 == T[k] is hit exactly.
- slot_fast_parts' conversion of d2 to float (clamp + funnel shift, restated in numpy) is
  truncation toward zero wherever it is not clamped.
- The classes mdh_rdf_bin_guess_audit enumerates cover every double >= 0, and the guess's
  float is constant on each.
- The host error bound of the guess: below the margin for every r_lo = 0 configuration of
  the GPU sweep, above it in the transition zone.
"""
import numpy as np
import pytest

import _threshold_pairs as tp

F32, F64 = np.float32, np.float64

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)


def _thr(n_bins, rr):
    from mdhelper_b200.analysis._binning import squared_thresholds
    return squared_thresholds(n_bins, rr)


def _rp():
    from oracle import reference_port as rp
    return rp


def _tri(shape, L):
    dims = np.array([L * shape[0], L * shape[1], L * shape[2], *shape[3:]], np.float32)
    return dims, _rp().triclinic_vectors(dims).astype(np.float32)


# (dims, cell or box, n_bins, range)
ORTHO = [
    ((16.0, 16.0, 16.0), 64, (0.0, 8.0)),            # dyadic: d2 == T[k] is hit
    ((11.0, 12.5, 13.25), 100, (1.0, 4.5)),          # r_lo > 0: T[0]
    ((650.0, 700.0, 710.0), 1000, (299.0, 300.0)),
]
TRI = [(RD, 20.0, 40, (0.0, 6.0)), (TO, 20.0, 40, (0.5, 6.0)), (TILT, 20.0, 60, (0.0, 5.0))]


def _cases():
    for box, n_bins, rr in ORTHO:
        b = np.array(box, np.float32)
        yield np.concatenate([b, [90, 90, 90]]).astype(np.float32), b, n_bins, rr
    for shape, L, n_bins, rr in TRI:
        dims, h = _tri(shape, L)
        yield dims, h, n_bins, rr


CASES = list(_cases())


def _assert_adjacent(c, p, k, above):
    """The two pairs of a threshold differ in one coordinate of one particle, by a few
    float32 steps: where the moved coordinate is the smaller of the two, several of its
    steps give the same float32 difference (straddle_pairs: per kind, the pairs below, then
    those above)."""
    starts = np.flatnonzero(np.diff(above.astype(int)) == 1) + 1       # below -> above
    ends = np.concatenate([np.flatnonzero(np.diff(above.astype(int)) == -1) + 1, [len(k)]])
    b0 = 0
    for s, e in zip(starts, ends):
        lo, hi = slice(b0, s), slice(s, e)
        assert s - b0 == e - s and np.array_equal(k[lo], k[hi])
        x = np.concatenate([c[lo], p[lo]], 1).view(np.int32).astype(np.int64)
        y = np.concatenate([c[hi], p[hi]], 1).view(np.int32).astype(np.int64)
        dx = np.abs(x - y)
        assert ((dx > 0).sum(1) == 1).all() and (dx.max(1) <= 8).all()
        b0 = e


def _oracle_slots(c, p, dims, n_bins, rr):
    """Per pair i (c[i], p[i]): the oracle's histogram slot (bin + 1; 0 / n_bins + 1 when not
    counted) and its distance (nan when not returned)."""
    rp = _rp()
    pairs, dist = rp.capped_distance(c, p, rr[1], rr[0] - np.finfo(F64).eps, box=dims,
                                     method="bruteforce")
    diag = pairs[:, 0] == pairs[:, 1]
    d = np.full(len(c), np.nan)
    d[pairs[diag, 0]] = dist[diag]
    slots = np.zeros(len(c), np.int64)
    got = ~np.isnan(d)
    edges = np.linspace(rr[0], rr[1], n_bins + 1)
    for i in np.flatnonzero(got):
        h = np.histogram([d[i]], bins=n_bins, range=rr)[0]
        slots[i] = int(np.argmax(h)) + 1 if h.sum() else 0
    # not returned by capped_distance: below r_lo or above r_hi
    slots[~got] = -1
    return slots, d, edges


@pytest.mark.parametrize("case", range(len(CASES)))
def test_straddling_pairs_land_where_the_oracle_puts_them(case):
    dims, box, n_bins, rr = CASES[case]
    rng = np.random.default_rng(case)
    thr = _thr(n_bins, rr)
    ks = tp.threshold_sample(n_bins, rng)
    c, p, d2, k, above = tp.straddle_pairs(box, thr, ks, rng)
    # every threshold of the sample is straddled (T[0] = 0 has nothing below it)
    want_ks = set(ks.tolist()) - ({0} if thr[0] == 0 else set())
    assert set(k.tolist()) == want_ks
    assert np.array_equal(d2, tp.ref_d2(c, p, box))
    assert (d2[above] >= thr[k[above]]).all() and (d2[~above] < thr[k[~above]]).all()
    _assert_adjacent(c, p, k, above)
    # the oracle: same slot, same distance bit for bit where it reports one
    want, dist, _ = _oracle_slots(c, p, dims, n_bins, rr)
    mine = np.searchsorted(thr, d2, side="right")
    counted = want > 0
    assert np.array_equal(mine[counted], want[counted])
    assert np.array_equal(np.sqrt(d2[counted]), dist[counted])
    assert ((mine[~counted] == 0) | (mine[~counted] == n_bins + 1)).all()
    # T[0] and T[n_bins]: the partner below T[0] / at or above T[n_bins] is not counted
    assert (mine[(k == 0) & ~above] == 0).all() if rr[0] > 0 else True
    assert (mine[(k == n_bins) & above] == n_bins + 1).all()
    assert (mine[(k == n_bins) & ~above] == n_bins).all()


def test_face_pairs_cross_the_periodic_face():
    box = np.array([11.0, 12.5, 13.25], np.float32)
    thr = _thr(100, (1.0, 4.5))
    rng = np.random.default_rng(3)
    c, p, d2, k, above = tp.straddle_pairs(box, thr, np.arange(101), rng, kinds=("face",))
    df = (p - c).astype(F64)
    assert (np.abs(df) > box / 2).any(1).all()                # the image shift is not zero
    tri = _tri(TO, 20.0)[1]
    c, p, d2, k, above = tp.straddle_pairs(tri, _thr(40, (0.0, 6.0)), np.arange(41), rng,
                                           kinds=("face",))
    dx = (tp.wrap(p, tri) - tp.wrap(c, tri)).astype(F64)
    assert (tp.image_d2(dx, tri, np.zeros_like(dx, dtype=np.int64)) > d2).all()


def test_dyadic_box_hits_the_thresholds_exactly():
    box = np.array([16.0, 16.0, 16.0], np.float32)
    thr = _thr(64, (0.0, 8.0))
    e2 = (np.arange(65) / 8.0) ** 2                            # the edges, squared: exact
    # T[k] <= edge^2 with the same square root; T[64] above 64: the last bin is closed
    assert (thr[:64] <= e2[:64]).all() and np.array_equal(np.sqrt(thr[:64]), np.arange(64) / 8)
    assert thr[64] > 64.0
    rng = np.random.default_rng(4)
    c, p, d2, k, above = tp.straddle_pairs(box, thr, np.arange(65), rng, kinds=("axis", "face"),
                                           grid=2.0 ** -8)
    # the partner at or above T[k] sits exactly on the edge: d2 == edge^2, the least d2 >= T[k]
    # the float32 inputs reach
    inner = above & (k < 64)
    assert np.array_equal(d2[inner], e2[k[inner]])
    assert len(set(k[inner].tolist())) >= 60


# ---- slot_fast_parts' float ------------------------------------------------------------------

def _trunc32(x):
    f = x.astype(F32)
    return np.where(f.astype(F64) > x, np.nextafter(f, F32(0)), f).astype(F32)


def _edge_doubles():
    e = []
    for k in range(-127, 129):
        t = np.ldexp(1.0, k)
        e += [t, np.nextafter(t, 0.0), np.nextafter(t, np.inf), 1.5 * t, 1.75 * t]
    f = np.random.default_rng(0).random(2000).astype(F32).astype(F64)
    e += list(f) + list(np.nextafter(f, 0.0)) + list(np.nextafter(f, 2.0))
    mid = f + np.ldexp(1.0, np.frexp(f)[1] - 25)                 # half an ulp above
    e += list(mid) + list(np.nextafter(mid, 0.0))
    return np.array(e, F64)


def test_truncation_trick_is_truncation_toward_zero():
    rng = np.random.default_rng(1)
    bits = rng.integers(0x3810000000000000, 0x47E0000000000000, 200000, dtype=np.int64)
    x = np.concatenate([bits.view(F64), _edge_doubles()])
    x = x[(x >= np.ldexp(1.0, -126)) & (x < np.ldexp(1.0, 127))]
    assert len(x) > 200000
    assert np.array_equal(tp.guess_float_bits(x), _trunc32(x).view(np.uint32))
    # below 2^-127: a float with a zero exponent, flushed to 0 by sqrt.approx.ftz
    small = np.concatenate([[0.0, 5e-324, 1e-300], np.ldexp(1.0, np.arange(-1074, -126)),
                            rng.integers(0, 0x3800000000000000, 10000).view(F64)])
    assert ((tp.guess_float_bits(small) & 0x7F800000) == 0).all()
    # 2^-127 <= x < 2^-126: hi word 0x380.....; the float is denormal as well
    assert ((tp.guess_float_bits(np.ldexp(1.0, -127) * 1.5) & 0x7F800000) == 0)
    # at and above 2^127, inf and NaN: clamped to [2^127, 2^127 (1 + 8 * 2^-23))
    big = np.concatenate([[np.ldexp(1.0, 127), 1e300, np.finfo(F64).max, np.inf, np.nan],
                          rng.integers(0x47E0000000000000, 0x7FF0000000000000, 10000).view(F64)])
    v = tp.guess_float_bits(big).view(F32).astype(F64)
    assert (v >= np.ldexp(1.0, 127)).all() and (v < np.ldexp(1.0 + 8 * 2.0 ** -23, 127)).all()


# ---- the audit's classes ----------------------------------------------------------------------

def test_classes_cover_every_nonnegative_double():
    rng = np.random.default_rng(2)
    bits = np.concatenate([
        rng.integers(0, 0x7FF0000000000000, 400000, dtype=np.int64),
        np.array([0, 1, 0x1FFFFFFF, 0x20000000, 0x37FFFFFFFFFFFFFF, 0x3800000000000000,
                  0x380000001FFFFFFF, 0x3800000020000000, 0x38000000FFFFFFFF,
                  0x3800000100000000, 0x47DFFFFFFFFFFFFF, 0x47E0000000000000,
                  0x47E00000FFFFFFFF, 0x47E0000100000000, 0x7FEFFFFFFFFFFFFF], np.int64)])
    x = bits.view(F64)
    c = tp.guess_class(x)
    assert (c >= 0).all() and (c < tp.N_CLASSES).all()
    lo, hi = tp.class_ends(c)
    u = bits.astype(np.uint64)
    assert ((lo <= u) & (u <= hi)).all()
    # the guess's float is the same at both ends of the class and in between
    g = tp.guess_float_bits(x)
    assert np.array_equal(g, tp.guess_float_bits(lo.view(F64)))
    assert np.array_equal(g, tp.guess_float_bits(hi.view(F64)))
    # classes are contiguous ranges of bit patterns, in order
    cs = np.unique(np.concatenate([rng.integers(0, tp.N_CLASSES - 1, 100000), [0, 7, 8],
                                   tp.N_CLASSES - 1 - np.arange(1, 9)]))
    _, hi_c = tp.class_ends(cs)
    lo_n, _ = tp.class_ends(cs + 1)
    # (the first and the last eight classes, hi word clamped, reach beyond their hi word)
    inner = (cs >= 7) & (cs <= tp.N_CLASSES - 9)
    assert np.array_equal(hi_c[inner] + np.uint64(1), lo_n[inner])
    # 0 opens the first class, the largest finite double closes the last; +inf (checked by
    # the audit separately) lies beyond it
    assert tp.class_ends(0)[0] == 0
    assert tp.class_ends(tp.N_CLASSES - 1)[1] == np.uint64(0x7FEFFFFFFFFFFFFF)
    assert tp.N_CLASSES == 2130706440


# ---- the host bound -------------------------------------------------------------------------

def test_host_bound_splits_the_sweep():
    ok = {}
    for r_lo, r_hi, n in tp.SWEEP:
        up, down, margin = tp.guess_error_bound(n, r_lo, r_hi)
        ok[(r_lo, r_hi, n)] = up < margin and down < 1 - margin
        if r_lo == 0:
            assert ok[(r_lo, r_hi, n)], (r_lo, r_hi, n, up, margin)
    assert ok[(49.0, 50.0, 1000)]
    for r in (100.0, 200.0, 300.0):
        up, _, margin = tp.guess_error_bound(1000, r - 1, r)
        assert up > margin, (r, up, margin)
    up, _, margin = tp.guess_error_bound(2000, 999.0, 1000.0)
    assert up > 10 * margin
    # configurations on both sides of the bound
    assert 5 <= sum(ok.values()) <= len(ok) - 5
    assert len(tp.SWEEP) >= 30
