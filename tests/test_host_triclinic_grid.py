"""CPU: the triclinic cell-list grid (mdh_rdf_triclinic_grid) and the single-image
argument behind rdf_tri_cells_kernel, restated in numpy with the operation order of the
kernels (rdf_tri.cu): for every pair whose 27-image minimum is in range, the stencil of
the planner's grid holds the partner exactly once, at an image whose d^2 equals the
minimum bit for bit."""
import numpy as np
import pytest

from _threshold_pairs import image_d2 as _image_d2, wrap as _wrap

U8 = 60          # kTriShiftMax


def _lib():
    from mdhelper_b200 import _lib
    return _lib


def _cell(dims):
    from mdhelper_b200.analysis._triclinic import triclinic_vectors
    return np.asarray(triclinic_vectors(np.asarray(dims, np.float32)), np.float32)


def _widths(h):
    h = h.astype(np.float64)
    a, b, c = h
    vol = abs(np.linalg.det(h))
    return np.array([vol / np.linalg.norm(np.cross(b, c)), vol / np.linalg.norm(np.cross(c, a)),
                     vol / np.linalg.norm(np.cross(a, b))])


def _tri_cell(p, h, nc):
    """tri_cell: fractional coordinates, cell per axis, lattice shift k = -floor(s)."""
    ax, bx, by, cx, cy, cz = (float(h[0, 0]), float(h[1, 0]), float(h[1, 1]), float(h[2, 0]),
                              float(h[2, 1]), float(h[2, 2]))
    x, y, z = (p[:, k].astype(np.float64) for k in range(3))
    sc = z / cz
    sb = (y - sc * cy) / by
    sa = ((x - sb * bx) - sc * cx) / ax
    c, k = [], []
    for s, n in zip((sa, sb, sc), nc):
        f = np.floor(s)
        c.append(np.clip(((s - f) * float(n)).astype(np.int64), 0, n - 1))
        k.append(np.clip(-f, -U8, U8).astype(np.int64))
    return np.stack(c, 1), np.stack(k, 1)


def _check(h, r_hi, p):
    nc, margin = _lib().triclinic_grid(h, r_hi, 10 ** 12)
    nc = np.array(nc)
    assert (nc >= 3).all(), (nc, margin)
    w = _widths(h)
    assert (w / nc >= r_hi + margin).all()
    U = r_hi * r_hi
    p = _wrap(p, h)
    cell, k = _tri_cell(p, h, nc)
    dx = (p[None, :, :] - p[:, None, :]).astype(np.float32).astype(np.float64)   # [i, j]
    m27 = np.array([(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)])
    min27 = np.full(dx.shape[:2], np.inf)
    for m in m27:
        min27 = np.minimum(min27, _image_d2(dx, h, np.broadcast_to(m, dx.shape)))
    # stencil: per axis the offsets d in {-1, 0, 1} with (c_i + d) mod n == c_j, and the
    # wrap w of c_i + d
    hits = np.ones(dx.shape[:2], np.int64)
    wrap = np.zeros(dx.shape, np.int64)
    for ax in range(3):
        n = nc[ax]
        ci, cj = cell[:, None, ax], cell[None, :, ax]
        cnt = np.zeros(dx.shape[:2], np.int64)
        for d in (-1, 0, 1):
            v = ci + d
            hit = (v % n) == cj
            cnt += hit
            wrap[..., ax] += np.where(hit, (v < 0) * -1 + (v >= n) * 1, 0)
        assert cnt.max() <= 1                       # distinct neighbour cells (n >= 3)
        hits *= cnt
    mprime = k[None, :, :] - k[:, None, :] + wrap
    in27 = (np.abs(mprime) <= 1).all(-1)
    d2s = _image_d2(dx, h, np.clip(mprime, -1, 1))
    near = min27 <= U
    assert near.sum() > len(p)                      # the cases do exercise the range
    # every pair in range is a candidate exactly once, at one of the 27 images
    assert (hits[near] == 1).all()
    assert in27[near].all()
    # the stencil image's d^2 is the 27-image minimum, bit for bit, when either is in range
    cand = (hits == 1) & in27
    either = cand & (near | (d2s <= U))
    assert np.array_equal(d2s[either].view(np.int64), min27[either].view(np.int64))
    # candidates at an image outside the 27 are out of range for the reference as well
    assert (min27[(hits == 1) & ~in27] > U).all()


def _adversarial(h, nc, r_hi, n_rand, rng):
    """Fractional coordinates 0, 1 - ulp, on cell faces and corners, plus partners at
    distances r_hi (1 +- small) across the periodic faces, plus random particles up to
    2 cells outside the box."""
    one_m = np.nextafter(1.0, 0.0)
    faces = [np.array([0.0, one_m, 0.5])] + [np.arange(n + 1) / n for n in nc]
    pts = []
    for _ in range(n_rand // 3):
        f = np.array([rng.choice(faces[1 + a]) if rng.random() < 0.6 else rng.random()
                      for a in range(3)])
        f = np.where(rng.random(3) < 0.2, rng.choice(faces[0], 3), f)
        pts.append(f @ h.astype(np.float64))
    pts = np.array(pts)
    u = rng.normal(size=(len(pts), 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    scale = r_hi * (1 + rng.choice([-1e-7, -1e-9, 0.0, 1e-9, 1e-7, -0.3], len(pts)))
    partners = pts + u * scale[:, None]
    rand = (rng.random((n_rand - 2 * len(pts), 3)) * 5 - 2) @ h.astype(np.float64)
    return np.concatenate([pts, partners, rand]).astype(np.float32)


CELLS = [
    (40.0, 40.0, 40.0, 60.0, 60.0, 90.0),              # rhombic dodecahedron
    (40.0, 40.0, 40.0, 70.53, 109.47, 70.53),          # truncated octahedron
    (30.0, 34.0, 38.0, 90.0, 118.0, 90.0),             # strongly tilted monoclinic
    (21.0, 22.5, 24.0, 75.0, 82.0, 64.0),
    (25.0, 25.0, 25.0, 60.0, 60.0, 60.0),
    (31.0, 29.0, 33.0, 115.0, 65.0, 120.0),
]


@pytest.mark.parametrize("dims", CELLS)
@pytest.mark.parametrize("rel", [0.33, 0.2, 0.05])
def test_single_image_is_the_27_image_minimum(dims, rel):
    rng = np.random.default_rng(abs(hash((dims, rel))) % 2 ** 32)
    h = _cell(dims)
    r_hi = rel * _widths(h).min()
    nc, _ = _lib().triclinic_grid(h, r_hi, 10 ** 12)
    _check(h, r_hi, _adversarial(h, nc, r_hi, 900, rng))


@pytest.mark.parametrize("dims", [CELLS[0], CELLS[1], CELLS[2]])
def test_large_cells_where_float32_rounding_of_dx_matters(dims):
    """L / r_hi about 150: |dx| up to the cell's extent, the float32 rounding of dx is
    no longer small against the relative slack alone."""
    rng = np.random.default_rng(7)
    h = _cell(np.array(dims) * np.array([3.75, 3.75, 3.75, 1, 1, 1]))   # edges 150 / 112..142
    r_hi = 1.0
    nc, margin = _lib().triclinic_grid(h, r_hi, 10 ** 12)
    assert min(nc) >= 60 and margin > 1e-5 * r_hi
    _check(h, r_hi, _adversarial(h, nc, r_hi, 900, rng))


def test_grid_limits_and_errors():
    L = _lib()
    h = _cell((30.0, 30.0, 30.0, 60.0, 60.0, 90.0))
    w = _widths(h)
    # exactly 3 cells on the narrowest axis; fewer than 3: no grid
    nc, m = L.triclinic_grid(h, w.min() / 3.2, 10 ** 12)
    assert min(nc) == 3
    assert L.triclinic_grid(h, w.min() / 2.9, 10 ** 12)[0] == (0, 0, 0)
    # at most 160 cells per axis, about 2 particles per cell
    assert max(L.triclinic_grid(h, 0.01, 10 ** 12)[0]) == 160
    nc, _ = L.triclinic_grid(h, 0.5, 2000)
    assert np.prod(nc) <= 1000 and min(nc) >= 3
    with pytest.raises(ValueError):                   # not lower triangular
        L.triclinic_grid(np.ones((3, 3), np.float32), 1.0, 100)
    with pytest.raises(ValueError):
        L.triclinic_grid(np.diag([1.0, 1.0, np.inf]).astype(np.float32), 1.0, 100)
