"""CPU: the fp32 evaluation of the triclinic cell list's filter, restated with every
operation rounded once (numpy float32 / float64 arithmetic is IEEE round-to-nearest; the
exact image in rationals), against its error bound (rdf_tri.cu::tri_cellq_kernel,
rdf_tri_cells_filter_kernel, tri_cells_filter_prepare; DESIGN.md 4.8c).

Checked on random and adversarial particles (cell faces and corners +- ulps, 1 - ulp,
partners at r (1 +- 1e-7)) in the oracle cells plus hexagonal, oblique and tilted-c cells:
  1. per axis, |u_f - u| <= A_k, u = dx + m' H the exact image of the candidate;
  2. the reference's d of the same image (float32 dx, fp64 sums and squares) differs from
     the fp32 d (sum of squares, sqrt) by at most the bound a plus the relative terms;
  3. candidates with m' outside {-1, 0, 1}^3 (truncated octahedron) exist and are the ones
     the image test sends to the scratch slot.
mdh_rdf_triclinic_cells_filter_window is checked against the restated eligibility."""
import math
from fractions import Fraction

import numpy as np
import pytest

from _threshold_pairs import image_d2

F32, F64 = np.float32, np.float64
E24, U53 = 2.0 ** -24, 2.0 ** -53

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)


def _scaled(shape, L):
    return (L * shape[0], L * shape[1], L * shape[2], *shape[3:])


CELLS = [(10.5, 11.25, 12.0, 75.0, 82.0, 64.0), (10.0, 11.5, 12.5, 90.0, 90.0, 70.0),
         (11.0, 11.0, 11.0, 60.0, 60.0, 60.0), _scaled(RD, 12.0), _scaled(TO, 12.0),
         _scaled(TILT, 12.0),
         (12.0, 12.0, 15.0, 90.0, 90.0, 120.0),          # hexagonal
         (12.0, 12.5, 13.0, 90.0, 90.0, 35.0),           # oblique (|b_x| > a_x / 2)
         (12.0, 12.0, 14.0, 62.0, 118.0, 90.0)]          # c tilted in x and y


def _cell(dims):
    from oracle import reference_port as rp
    return rp.triclinic_vectors(np.array(dims, np.float32)).astype(F32)


def _rows(h):
    h = h.astype(F64)
    return np.array([h[0, 0] + abs(h[1, 0]) + abs(h[2, 0]), h[1, 1] + abs(h[2, 1]), h[2, 2]])


def _A(h):
    """tri_cells_filter_prepare: the per-axis bound A_k and a."""
    h64 = h.astype(F64)
    R = _rows(h)
    E = np.array([h64[0, 0], h64[1, 1], h64[2, 2]])
    Q = R * (1 + 1e-9)
    eq = E24 * Q + 3 * U53 * (1.5 * E + 60 * R)
    ev = E24 * (R + Q) * (1 + 2 * E24) + 3 * U53 * (R + Q)
    Ak = 2 * eq + ev
    ax, bx, by, cx, cy, cz = h64[0, 0], h64[1, 0], h64[1, 1], h64[2, 0], h64[2, 1], h64[2, 2]
    rows = np.array([3 * ax + abs(bx) + abs(cx), 3 * by + abs(cy), 3 * cz])
    e_f = 2 * np.linalg.norm(E) * E24
    e_d = 4 * U53 * np.linalg.norm(rows)
    a = (np.linalg.norm(Ak) * (1 + 1e-9) + e_f + e_d) * (1 + 1e-9)
    return Ak, a


def _kshift(r, h):
    """tri_cell: fractional coordinates in fp64, k = -floor(s) per axis."""
    h = h.astype(F64)
    x, y, z = (r[:, k].astype(F64) for k in range(3))
    sc = z / h[2, 2]
    sb = (y - sc * h[2, 1]) / h[1, 1]
    sa = ((x - sb * h[1, 0]) - sc * h[2, 0]) / h[0, 0]
    return -np.floor(np.stack([sa, sb, sc], 1))


def _q(r, k, h):
    """tri_cellq_kernel: q = r + k H, fp64 sums, one float32 rounding."""
    h = h.astype(F64)
    x, y, z = (r[:, i].astype(F64) for i in range(3))
    qx = ((x + k[:, 0] * h[0, 0]) + k[:, 1] * h[1, 0]) + k[:, 2] * h[2, 0]
    qy = (y + k[:, 1] * h[1, 1]) + k[:, 2] * h[2, 1]
    qz = z + k[:, 2] * h[2, 2]
    return np.stack([qx, qy, qz], 1).astype(F32)


def _wrapped_particles(h, n, rng, r_hi):
    """Wrapped particles: random, at faces and corners +- ulps and at 1 - ulp, plus
    partners at r_hi (1 +- 1e-7) in random directions (wrapped back into the brick)."""
    h64 = h.astype(F64)
    one_m = np.nextafter(1.0, 0.0)
    spots = np.array([0.0, 1e-7, 0.5, one_m, 1.0 - 1e-7])
    fr = np.concatenate([rng.random((n, 3)),
                         np.stack(np.meshgrid(spots, spots, spots), -1).reshape(-1, 3)])
    base = (fr @ h64).astype(F32)
    base = np.concatenate([base, np.nextafter(base, F32(np.inf)),
                           np.nextafter(base, F32(-np.inf))])
    v = rng.normal(size=base.shape)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    lens = r_hi * rng.choice([1 - 1e-7, 1.0, 1 + 1e-7, 0.5, 0.999], len(base))[:, None]
    partner = (base.astype(F64) + v * lens).astype(F32)
    # wrapped coordinates lie in the brick [-E/2, 3E/2] of a non-far frame
    E = np.array([h64[0, 0], h64[1, 1], h64[2, 2]])
    partner = np.clip(partner, (-0.5 * E).astype(F32), (1.5 * E).astype(F32))
    return base, partner


def _evaluate(h, ri, rj, flat=False):
    """Per candidate: m' (for w = 0 here: m' = k_j - k_i), the fp32 u and d, the exact u."""
    ki, kj = _kshift(ri, h), _kshift(rj, h)
    if flat:
        ki[:, 2] = kj[:, 2] = 0
    qi, qj = _q(ri, ki, h), _q(rj, kj, h)
    m = kj - ki
    # w: the wrap code; any w gives the same image m' = k_j - k_i + w; use w = m - (k_j - k_i)
    # = 0 and compute v in fp64 as the kernel does
    v = (0.0 - qi.astype(F64)).astype(F32)
    u = (qj + v).astype(F32)
    # fma(uz, uz, fma(uy, uy, ux * ux)): the products are exact in fp64
    u64 = u.astype(F64)
    t = (u[:, 0] * u[:, 0]).astype(F32)
    t = (u64[:, 1] * u64[:, 1] + t.astype(F64)).astype(F32)
    d2 = (u64[:, 2] * u64[:, 2] + t.astype(F64)).astype(F32)
    return m, u, d2


@pytest.mark.parametrize("dims", CELLS, ids=range(len(CELLS)))
def test_per_axis_bound_and_reference_gap(dims):
    rng = np.random.default_rng(int(sum(dims) * 10))
    h = _cell(dims)
    h64 = h.astype(F64)
    r_hi = 2.5
    ri, rj = _wrapped_particles(h, 200, rng, r_hi)
    m, u, d2 = _evaluate(h, ri, rj)
    Ak, a = _A(h)
    # 1. per axis, against the exact image dx + m' H in rationals (on a sample)
    H = [[Fraction(float(h64[r, c])) for c in range(3)] for r in range(3)]
    for t in rng.choice(len(ri), 150, replace=False):
        for ax in range(3):
            exact = Fraction(float(rj[t, ax])) - Fraction(float(ri[t, ax]))
            exact += sum(int(m[t, r]) * H[r][ax] for r in range(3))
            assert abs(Fraction(float(u[t, ax])) - exact) <= Fraction(Ak[ax]), (t, ax)
    # 2. the reference's d of the same image, where m' is one of its 27
    ok = np.all(np.abs(m) <= 1, axis=1)
    dx = (rj - ri).astype(F32).astype(F64)
    dref = np.sqrt(image_d2(dx[ok], h, m[ok].astype(int)))
    df = np.sqrt(d2[ok].astype(F64))
    gap = np.abs(df - dref)
    lim = a + (2.5 * E24 * 1.001 + 4 * U53) * np.maximum(df, dref) + 1e-12
    assert np.all(gap <= lim), float(np.max(gap - lim))


def test_flat_grid_c_one_ulp_above():
    """drop_axis = 2: z = 0, k_c = 0, q_z = u_z = 0; c_z one ulp above r + M."""
    from mdhelper_b200 import _lib
    rng = np.random.default_rng(3)
    h = _cell((12.0, 12.0, 15.0, 90.0, 90.0, 120.0))
    r_hi = 2.5
    _, margin = _lib.triclinic_grid(h, r_hi, 1000)
    h[2, 2] = np.nextafter(F32(r_hi + margin), F32(np.inf))
    ri, rj = _wrapped_particles(h, 200, rng, r_hi)
    ri[:, 2] = 0.0
    rj[:, 2] = 0.0
    m, u, d2 = _evaluate(h, ri, rj, flat=True)
    assert np.all(m[:, 2] == 0) and np.all(u[:, 2] == 0)
    _, a = _A(h)
    ok = np.all(np.abs(m) <= 1, axis=1)
    dx = (rj - ri).astype(F32).astype(F64)
    dref = np.sqrt(image_d2(dx[ok], h, m[ok].astype(int)))
    df = np.sqrt(d2[ok].astype(F64))
    assert np.all(np.abs(df - dref) <= a + 3 * E24 * np.maximum(df, dref))


def test_truncated_octahedron_images_outside_the_27():
    """Some candidates of a truncated octahedron have m' outside {-1, 0, 1}^3; the kernel's
    per-byte test (VADD4 / VCMPLEU4) flags exactly those."""
    rng = np.random.default_rng(4)
    h = _cell(_scaled(TO, 12.0))
    ri, rj = _wrapped_particles(h, 2000, rng, 5.0)
    # shift the partners by lattice vectors so that m' reaches +-2
    rj = (rj.astype(F64) + np.array([1, -1, 1]) @ h.astype(F64)).astype(F32)
    m = _kshift(rj, h) - _kshift(ri, h)
    code = np.zeros(len(m), np.uint32)
    for ax in range(3):
        code |= (m[:, ax].astype(np.int64) & 0xff).astype(np.uint32) << (8 * ax)
    # __vadd4 adds per byte without carries, __vcmpleu4 compares per byte
    bytes_ok = np.all([(((code >> (8 * b)) & 0xff) + 1) % 256 <= 2 for b in range(3)], axis=0)
    want = np.all(np.abs(m) <= 1, axis=1)
    assert (~want).any() and want.any()
    assert np.array_equal(bytes_ok, want)


def _mu(h, n_bins, r_lo, r_hi, sqrt_err, k):
    _, a = _A(h)
    scale = n_bins / (r_hi - r_lo)
    d_max = r_hi + 2.0 / scale
    return (scale * (a + d_max * (2.5 * E24 * 1.001 + sqrt_err + 4 * U53)) +
            E24 * scale * d_max * 1.001 + 1.0 / 2 ** k + 1e-9)


@pytest.mark.parametrize("n_bins,r_lo,r_hi", [(100, 0.0, 2.5), (1000, 0.0, 2.5),
                                              (40, 1.0, 3.0), (7, 0.0, 3.0)])
def test_window_entry_point_matches_the_restated_eligibility(n_bins, r_lo, r_hi):
    from mdhelper_b200 import _lib
    cells = np.stack([_cell(d) for d in CELLS] + [_cell(_scaled(RD, 5000.0))])
    win = _lib.triclinic_cells_filter_window(n_bins, r_lo, r_hi, cells, sqrt_err=2.0 ** -22)
    for h, w in zip(cells, win):
        k = w["k"]
        mu = _mu(h, n_bins, r_lo, r_hi, 2.0 ** -22, k)
        assert math.isclose(w["mu"], mu, rel_tol=1e-12)
        m = math.ceil(1.25 * mu * 2 ** k) + 1
        eligible = m >= 1 and 2 * m + 1 < 2 ** k / 8
        assert w["eligible"] == int(eligible)
        if eligible:
            assert w["wlim"] == 2 * m + 1
    # a huge cell: the bound is not small against a bin, the frame is declined
    assert win[-1]["eligible"] == 0 or n_bins < 1000


def test_window_entry_point_rejects_invalid_input():
    from mdhelper_b200 import _lib
    h = _cell(_scaled(RD, 12.0))
    bad = h.copy()
    bad[0, 1] = 1.0                                  # not lower triangular
    with pytest.raises(ValueError):
        _lib.triclinic_cells_filter_window(10, 0.0, 2.5, bad[None])
    with pytest.raises(ValueError):
        _lib.triclinic_cells_filter_window(10, 2.5, 1.0, h[None])
