"""CPU: the sheared fp32 fold of the triclinic RDF filter, restated in float32 with every
FMA rounded once from exact rationals (rdf_tri.cu::tri_fold2, tri_filter_prepare_frame;
DESIGN.md 4.8b).

The claims checked against exact arithmetic and the reference's 27-image fp64 minimum
(_threshold_pairs.tri_ref_d2), on random pairs and on adversarial ones (brick faces and
corners +- a few ulps, |u| at R +- ulps, fold indices of 2):
  1. the exact folded image u = df - n_c c - n_b b - n_a a lies within delta of the brick B
     (half-widths a_x/2, b_y/2, c_z/2); when |u| < R = min(a_x, b_y, c_z)/2 it is the
     shortest image of df over a +-3 lattice neighbourhood;
  2. per axis, |u_f - u| is within the fold's error bound; when |u| < R and every |n_k| <= 1,
     the reference's 27-image d differs from |u_f| by at most the bound a of the window;
     when |u| < R and some |n_k| >= 2, the reference's d is at least R - (its fp64 error);
  3. the true minimum is at least min(|u|, R - delta).
mdh_rdf_triclinic_filter_window is checked against the restated eligibility, and to decline
frames with inf / NaN / huge extents and with r_hi >= R."""
import math
from fractions import Fraction

import numpy as np
import pytest

from _threshold_pairs import tri_ref_d2, wrap

F32 = np.float32
E24 = 2.0 ** -24
U53 = 2.0 ** -53
MAGIC = F32(12582912.0)

RD = (1.0, 1.0, 1.0, 60.0, 60.0, 90.0)
TO = (1.0, 1.0, 1.0, 70.53, 109.47, 70.53)
TILT = (1.0, 1.1, 1.2, 90.0, 118.0, 90.0)


def _scaled(shape, L):
    return (L * shape[0], L * shape[1], L * shape[2], *shape[3:])


CELLS = [(10.5, 11.25, 12.0, 75.0, 82.0, 64.0), (10.0, 11.5, 12.5, 90.0, 90.0, 70.0),
         (11.0, 11.0, 11.0, 60.0, 60.0, 60.0), _scaled(RD, 12.0), _scaled(TO, 12.0),
         _scaled(TILT, 12.0),
         (12.0, 12.0, 15.0, 90.0, 90.0, 120.0),          # hexagonal
         (12.0, 12.5, 13.0, 90.0, 90.0, 35.0)]           # unreduced tilt (|b_x| > a_x / 2)


def _cell(dims):
    from oracle import reference_port as rp
    return rp.triclinic_vectors(np.array(dims, np.float32)).astype(F32)


def f32(q):
    """Round the rational q to the nearest float32 (ties to even)."""
    c = F32(float(q))
    best = None
    for v in (np.nextafter(c, F32(-np.inf)), c, np.nextafter(c, F32(np.inf))):
        d = abs(Fraction(float(v)) - q)
        if best is None or d < best[0] or (d == best[0] and
                                           (int(np.array(v).view(np.uint32)) & 1) == 0):
            best = (d, v)
    return F32(best[1])


def fma(a, b, c):
    return f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def fold(df, h):
    """tri_fold2 for one pair: n (float32 integers), u_f (float32), |u_f|^2 in float32."""
    inv = [F32(1.0 / float(h[0, 0])), F32(1.0 / float(h[1, 1])), F32(1.0 / float(h[2, 2]))]
    nc = f32(Fraction(float(fma(df[2], inv[2], MAGIC))) - Fraction(float(MAGIC)))
    uz = fma(nc, -h[2, 2], df[2])
    y1 = fma(nc, -h[2, 1], df[1])
    x1 = fma(nc, -h[2, 0], df[0])
    nb = f32(Fraction(float(fma(y1, inv[1], MAGIC))) - Fraction(float(MAGIC)))
    uy = fma(nb, -h[1, 1], y1)
    x2 = fma(nb, -h[1, 0], x1)
    na = f32(Fraction(float(fma(x2, inv[0], MAGIC))) - Fraction(float(MAGIC)))
    ux = fma(na, -h[0, 0], x2)
    return (int(na), int(nb), int(nc)), np.array([ux, uy, uz], F32)


def bounds(h, D):
    """The per-axis fold error, delta_k and the reference's fp64 error of
    tri_filter_prepare_frame for extents D of |df|."""
    ax, bx, by, cx, cy, cz = (float(h[0, 0]), float(h[1, 0]), float(h[1, 1]), float(h[2, 0]),
                              float(h[2, 1]), float(h[2, 2]))
    ia, ib, ic = float(F32(1 / ax)), float(F32(1 / by)), float(F32(1 / cz))
    ea, eb, ec = abs(ia * ax - 1), abs(ib * by - 1), abs(ic * cz - 1)
    Nc = math.floor(D[2] * ic * (1 + 1e-12) + 0.5)
    Y1 = (D[1] + Nc * abs(cy)) * (1 + E24)
    Nb = math.floor(Y1 * ib * (1 + 1e-12) + 0.5)
    X1 = (D[0] + Nc * abs(cx)) * (1 + E24)
    X2 = (X1 + Nb * abs(bx)) * (1 + E24)
    d = np.array([X2 * ea + E24 * (X1 + X2), Y1 * (eb + E24), D[2] * ec]) * (1 + 1e-6)
    H = np.array([ax, by, cz]) / 2 + d
    f = np.array([E24 * (X1 + X2 + H[0]), E24 * (Y1 + H[1]), E24 * H[2]]) * (1 + 1e-6)
    r = np.array([3 * U53 * (D[0] + ax + abs(bx) + abs(cx)), 2 * U53 * (D[1] + by + abs(cy)),
                  U53 * (D[2] + cz)])
    return f, d, r


def exact_u(df, n, h):
    H = [[Fraction(float(h[r, k])) for k in range(3)] for r in range(3)]
    return [Fraction(float(df[k])) - n[2] * H[2][k] - n[1] * H[1][k] - n[0] * H[0][k]
            for k in range(3)]


def shortest(df, h, reach=3):
    """Exact squared length of the shortest image over a +-reach neighbourhood."""
    H = [[Fraction(float(h[r, k])) for k in range(3)] for r in range(3)]
    best = None
    rng_ = range(-reach, reach + 1)
    for i in rng_:
        for j in rng_:
            for k in rng_:
                v = [Fraction(float(df[a])) + i * H[0][a] + j * H[1][a] + k * H[2][a]
                     for a in range(3)]
                s = sum(x * x for x in v)
                best = s if best is None or s < best else best
    return best


def _pairs(h, rng, n_random=40):
    """Wrapped coordinates in the brick [0, a_x) x [0, b_y) x [0, c_z): random pairs, pairs
    whose fold arguments sit on half-integers +- ulps (brick faces and corners), |u| = R +-
    ulps and fold indices of 2."""
    E = np.array([h[0, 0], h[1, 1], h[2, 2]], np.float64)
    hd = h.astype(np.float64)
    R = 0.5 * E.min()
    P = []
    for _ in range(n_random):
        P.append((rng.random(3) * E, rng.random(3) * E))
    for _ in range(12):
        # u on a brick face or corner: df = u + m H with u_k = +-E_k / 2 for some axes
        u = (rng.random(3) - 0.5) * E
        for k in np.nonzero(rng.random(3) < 0.6)[0]:
            u[k] = 0.5 * E[k] * rng.choice([-1, 1])
        m = rng.integers(-1, 2, 3)
        df = u + m @ hd
        xi = np.clip(rng.random(3) * E, 0, E)
        for s in (-3, -1, 0, 1, 3):
            xj = F32(xi + df) + F32(s) * np.spacing(F32(xi + df))
            P.append((xi, xj))
    for s in (-2, 0, 2):
        # |u| = R +- ulps along the shortest axis
        k = int(np.argmin(E))
        u = np.zeros(3)
        u[k] = R
        xi = 0.25 * E
        xj = F32(xi + u) + F32(s) * np.spacing(F32(xi + u))
        P.append((xi, xj))
    for _ in range(6):
        # a fold index of 2: in the truncated octahedron u = (-0.345, 0.015, -0.01) a_x is
        # the shortest image of u + 2a - b + c, a difference of two points of the brick
        u = np.array([-0.345, 0.015, -0.01]) * E[0] + 0.002 * rng.random(3) * E
        df = u + np.array([2, -1, 1]) @ hd
        xi = np.array([0.005, 0.504, 0.006]) * E + 0.002 * rng.random(3) * E
        P.append((xi, xi + df))
    return [(F32(np.asarray(a, F32)), F32(np.asarray(b, F32))) for a, b in P]


@pytest.mark.parametrize("dims", CELLS, ids=range(len(CELLS)))
def test_fold_claims(dims):
    h = _cell(dims)
    hd = h.astype(np.float64)
    rng = np.random.default_rng(11)
    E = np.array([h[0, 0], h[1, 1], h[2, 2]], np.float64)
    R = Fraction(float(E.min())) / 2
    n2 = 0
    for xi, xj in _pairs(h, rng):
        # the kernel and the reference both take differences of wrapped coordinates
        xi, xj = wrap(np.asarray(xi, F32)[None], h)[0], wrap(np.asarray(xj, F32)[None], h)[0]
        df = (xj - xi).astype(F32)
        D = np.abs(df.astype(np.float64)) * (1 + 2 * E24)
        f, d, r = bounds(h, D)
        n, uf = fold(df, h)
        u = exact_u(df, n, h)
        # fold error per axis and delta
        for k in range(3):
            assert abs(Fraction(float(uf[k])) - u[k]) <= Fraction(float(f[k])), (dims, k)
            assert abs(u[k]) <= Fraction(float(E[k])) / 2 + Fraction(float(d[k])), (dims, k)
        u2 = sum(x * x for x in u)
        delta = Fraction(float(d.max()))
        true2 = shortest(df, h)
        # claim 3: the true minimum is at least min(|u|, R - delta)
        lo = min(u2, (R - delta) ** 2)
        assert true2 >= lo * (1 - Fraction(1, 10 ** 12)), dims
        if u2 < R * R:
            # claim 1: u is the shortest image
            assert true2 == u2, dims
            ref = float(tri_ref_d2(xi[None], xj[None], hd.astype(F32))[0])
            if max(abs(v) for v in n) <= 1:
                # claim 2: |u_f| against the reference's d of the same image
                a = float(np.linalg.norm(f + r)) + math.sqrt(ref) * 4 * U53
                assert abs(float(np.linalg.norm(uf.astype(np.float64))) - math.sqrt(ref)) <= a
            else:
                n2 += 1
                assert math.sqrt(ref) >= float(R) * (1 - 1e-12) - float(np.linalg.norm(r))
    if dims in (_scaled(TO, 12.0),):
        assert n2 > 0


def _window_restated(h, ext, r_lo, r_hi, n_bins, sqrt_err=2.0 ** -22):
    D = np.maximum(np.maximum(ext[3:] - ext[:3], 0.0), 0.0).astype(np.float64) * (1 + 2 * E24)
    f, d, r = bounds(h, D)
    a = float(np.linalg.norm(f + r))
    scale = n_bins / (r_hi - r_lo)
    d_max = r_hi + 2 / scale
    lg = 0
    while (1 << lg) < n_bins + 2:
        lg += 1
    k = min(16, 22 - lg)
    mu = scale * (a + d_max * (1.5 * E24 * 1.001 + sqrt_err + 4 * U53)) + \
        E24 * scale * d_max * 1.001 + 2.0 ** -k + 1e-9
    R = 0.5 * float(min(h[0, 0], h[1, 1], h[2, 2]))
    reach = d_max + 1.25 * mu / scale + 2 * (float(np.linalg.norm(r)) + 4 * U53 * R) + d.max()
    m = math.ceil(1.25 * mu * 2 ** k) + 1
    return int(reach * (1 + 1e-9) < R and 2 * m + 1 < 2 ** k / 8), 2 * m + 1, R


@pytest.mark.parametrize("dims", CELLS, ids=range(len(CELLS)))
def test_window_entry(dims):
    from mdhelper_b200 import _lib
    h = _cell(dims)
    E = np.array([h[0, 0], h[1, 1], h[2, 2]], F32)
    ext = np.concatenate([np.zeros(3, F32), E]).astype(F32)
    R = 0.5 * float(E.min())
    for r_hi in (0.5 * R, 0.9 * R, 0.999 * R, R, 1.2 * R):
        w = _lib.triclinic_filter_window(100, 0.0, r_hi, h[None], ext[None])[0]
        elig, wlim, Rr = _window_restated(h, ext, 0.0, r_hi, 100)
        assert w["eligible"] == elig and abs(w["R"] - Rr) < 1e-12 * Rr
        if elig:
            assert w["wlim"] == wlim
        if r_hi >= R:
            assert w["eligible"] == 0
    assert _lib.triclinic_filter_window(100, 0.0, 0.5 * R, h[None], ext[None])[0]["eligible"]
    for bad in (np.inf, np.nan, 3.0e8 * float(E[0])):
        e = ext.copy()
        e[3] = bad
        assert _lib.triclinic_filter_window(100, 0.0, 0.5 * R, h[None], e[None])[0][
            "eligible"] == 0
