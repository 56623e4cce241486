"""CPU: the cell-list grids of two-dimensional RDFs (drop_axis) from mdh_rdf_cells_grid, and
the single-image argument behind the flat triclinic grid (drop_axis = 2), restated in numpy
with the operation order of the kernels (rdf_tri.cu): particles with z zeroed and wrapped lie
in the (a, b) plane, and for every pair whose 27-image minimum is in range the 9-cell
stencil of the plane holds the partner exactly once, at an image whose d^2 equals the
minimum bit for bit."""
import numpy as np
import pytest

U8 = 60          # kTriShiftMax


def _lib():
    from mdhelper_b200 import _lib
    return _lib


def _cell(dims):
    from mdhelper_b200.analysis._triclinic import triclinic_vectors
    return np.asarray(triclinic_vectors(np.asarray(dims, np.float32)), np.float32)


def _widened(dims, drop):
    """The reference's two-dimensional cell: the dropped edge becomes the longest edge."""
    d = np.asarray(dims, np.float32).copy()
    d[drop] = d[:3].max()
    return d


def _plane_widths(h):
    """Line spacings of the (a, b) lattice in the plane z = 0: a_x b_y / |b| and b_y."""
    h = h.astype(np.float64)
    return np.array([h[0, 0] * h[1, 1] / np.hypot(h[1, 0], h[1, 1]), h[1, 1]])


# ---- orthorhombic grids ---------------------------------------------------------------------

@pytest.mark.parametrize("drop", [0, 1, 2])
@pytest.mark.parametrize("edges,r_hi,n_max", [((30.0, 40.0, 50.0), 2.5, 200_000),
                                              ((9.1, 9.4, 9.7), 3.0, 1000),
                                              ((800.0, 700.0, 20.0), 2.5, 500_000),
                                              ((60.0, 61.0, 62.0), 1.0, 2000)])
def test_orthorhombic_grid_has_one_cell_on_the_dropped_axis(drop, edges, r_hi, n_max):
    L = _lib()
    h = np.diag(_widened(list(edges) + [90, 90, 90], drop)[:3]).astype(np.float32)
    nc, margin = L.cells_grid(h, r_hi, n_max, drop)
    nc = np.array(nc)
    keep = [k for k in range(3) if k != drop]
    assert nc[drop] == 1
    assert (nc[keep] >= 3).all() and (nc[keep] <= 160).all()
    box = np.diag(h).astype(np.float64)
    assert (box[keep] / nc[keep] >= r_hi * 1.00001).all()
    assert margin == pytest.approx(1e-5 * r_hi)
    # about 2 particles per cell over the plane, unless the kept axes are down to 3 cells
    assert nc.prod() <= max(9, n_max / 2) or nc[keep].max() == 3
    # no kept axis could take a cell more without passing the cap or the occupancy rule
    for k in keep:
        more = nc.copy()
        more[k] += 1
        assert (more[k] > 160 or box[k] / more[k] < r_hi * 1.00001
                or more.prod() > max(9, n_max / 2)), (k, nc)


def test_orthorhombic_grid_without_drop_is_the_three_dimensional_one():
    L = _lib()
    h = np.diag([21.0, 23.5, 22.25]).astype(np.float32)
    nc, _ = L.cells_grid(h, 2.5, 6001)
    assert min(nc) >= 3 and np.prod(nc) <= max(27, 6001 / 2)
    # fewer than 3 cells on a kept axis: no grid; on the dropped axis it does not matter
    h = np.diag([30.0, 30.0, 7.0]).astype(np.float32)
    assert L.cells_grid(h, 2.5, 10_000) == ((0, 0, 0), pytest.approx(2.5e-5))
    assert L.cells_grid(h, 2.5, 10_000, 2)[0][2] == 1


# ---- triclinic grids --------------------------------------------------------------------------

HEX120 = (30.0, 30.0, 30.0, 90.0, 90.0, 120.0)
HEX60 = (40.0, 40.0, 25.0, 90.0, 90.0, 60.0)
TILTED_C = (30.0, 34.0, 22.0, 75.0, 108.0, 90.0)        # c tilted out of the normal
OBLIQUE = (31.0, 29.0, 33.0, 115.0, 65.0, 120.0)
FLAT_CELLS = [HEX120, HEX60, TILTED_C, OBLIQUE]


@pytest.mark.parametrize("dims", FLAT_CELLS)
@pytest.mark.parametrize("rel,n_max", [(0.33, 10 ** 12), (0.05, 10 ** 12), (0.02, 3000)])
def test_flat_triclinic_grid(dims, rel, n_max):
    L = _lib()
    h = _cell(_widened(dims, 2))
    w = _plane_widths(h)
    r_hi = rel * w.min()
    nc, margin = L.cells_grid(h, r_hi, n_max, 2)
    assert nc[2] == 1 and min(nc[:2]) >= 3 and max(nc[:2]) <= 160
    assert (w / np.array(nc[:2]) >= r_hi + margin).all()
    assert h[2, 2] >= r_hi + margin
    assert 1e-5 * r_hi <= margin < 1e-3 * r_hi + 1e-4
    assert np.prod(nc) <= max(9, n_max / 2) or min(nc[:2]) == 3
    # the 3-D planner is what drop_axis=None gets
    assert L.cells_grid(h, r_hi, n_max) == L.triclinic_grid(h, r_hi, n_max)


def test_triclinic_grid_errors():
    L = _lib()
    h = _cell(HEX120)
    for drop in (0, 1):
        with pytest.raises(ValueError, match="drop_axis 2"):
            L.cells_grid(h, 2.0, 1000, drop)
    # c_z below r_hi + M: no flat grid, although 3 cells fit in the plane
    thin = np.array([[30, 0, 0], [-15, 26, 0], [12, 9, 5]], np.float32)
    assert L.cells_grid(thin, 4.9, 1000, 2)[0][2] == 1
    with pytest.raises(ValueError, match="c_z"):
        L.cells_grid(thin, 5.0, 1000, 2)
    with pytest.raises(ValueError, match="c_z"):
        L.cells_grid(thin, 6.0, 1000, 2)
    # fewer than 3 cells in the plane: no grid
    assert L.cells_grid(h, 0.34 * _plane_widths(h).min(), 1000, 2)[0] == (0, 0, 0)
    with pytest.raises(ValueError):
        L.cells_grid(h, 1.0, 1000, 3)
    with pytest.raises(ValueError):
        L.cells_grid(np.ones((3, 3), np.float32), 1.0, 100, 2)


# ---- the one-image argument, pair by pair -----------------------------------------------------

def _wrap(p, h):
    """tri_wrap_kernel: along c, then b, then a, in double, rounded to float32."""
    ax, bx, by, cx, cy, cz = (float(h[0, 0]), float(h[1, 0]), float(h[1, 1]), float(h[2, 0]),
                              float(h[2, 1]), float(h[2, 2]))
    x, y, z = (p[:, k].astype(np.float64) for k in range(3))
    s = np.floor(z / cz)
    x, y, z = x - s * cx, y - s * cy, z - s * cz
    s = np.floor(y / by)
    x, y = x - s * bx, y - s * by
    x = x - np.floor(x / ax) * ax
    return np.stack([x, y, z], 1).astype(np.float32)


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


def _image_d2(dx, h, m):
    """tri_image_d2 with the shift terms h_k * i."""
    h = h.astype(np.float64)
    ix, iy, iz = (m[..., k].astype(np.float64) for k in range(3))
    rx = ((dx[..., 0] + h[0, 0] * ix) + h[1, 0] * iy) + h[2, 0] * iz
    ry = (dx[..., 1] + h[1, 1] * iy) + h[2, 1] * iz
    rz = dx[..., 2] + h[2, 2] * iz
    return (rx * rx + ry * ry) + rz * rz


def _check_flat(h, r_hi, p):
    nc, margin = _lib().cells_grid(h, r_hi, 10 ** 12, 2)
    nc = np.array(nc)
    assert nc[2] == 1 and (nc[:2] >= 3).all(), (nc, margin)
    U = r_hi * r_hi
    p = p.copy()
    p[:, 2] = 0.0                                   # rdf_pack_kernel, before the wrap
    p = _wrap(p, h)
    assert (p[:, 2] == 0).all()                     # the wrap keeps the plane
    cell, k = _tri_cell(p, h, nc)
    assert (cell[:, 2] == 0).all() and (k[:, 2] == 0).all()
    dx = (p[None, :, :] - p[:, None, :]).astype(np.float32).astype(np.float64)   # [i, j]
    m27 = np.array([(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)])
    min27 = np.full(dx.shape[:2], np.inf)
    for m in m27:
        min27 = np.minimum(min27, _image_d2(dx, h, np.broadcast_to(m, dx.shape)))
    # stencil: per kept axis the offsets d in {-1, 0, 1} with (c_i + d) mod n == c_j and the
    # wrap w of c_i + d; along c only d = 0 (one cell, no wrap)
    hits = np.ones(dx.shape[:2], np.int64)
    wrap = np.zeros(dx.shape, np.int64)
    for ax in range(2):
        n = nc[ax]
        ci, cj = cell[:, None, ax], cell[None, :, ax]
        cnt = np.zeros(dx.shape[:2], np.int64)
        for d in (-1, 0, 1):
            v = ci + d
            hit = (v % n) == cj
            cnt += hit
            wrap[..., ax] += np.where(hit, (v < 0) * -1 + (v >= n) * 1, 0)
        assert cnt.max() <= 1
        hits *= cnt
    mprime = k[None, :, :] - k[:, None, :] + wrap
    assert (mprime[..., 2] == 0).all()
    in27 = (np.abs(mprime) <= 1).all(-1)
    d2s = _image_d2(dx, h, np.clip(mprime, -1, 1))
    near = min27 <= U
    assert near.sum() > len(p)                      # the cases do exercise the range
    assert (hits[near] == 1).all()
    assert in27[near].all()
    cand = (hits == 1) & in27
    either = cand & (near | (d2s <= U))
    assert np.array_equal(d2s[either].view(np.int64), min27[either].view(np.int64))
    assert (min27[(hits == 1) & ~in27] > U).all()


def _adversarial(h, nc, r_hi, n_rand, rng):
    """In-plane fractional coordinates 0, 1 - ulp, on cell faces and corners, partners at
    distances r_hi (1 +- 1e-7 ...) in the plane and across the periodic faces, and random
    particles up to 2 cells outside the box (any z: it is zeroed)."""
    one_m = np.nextafter(1.0, 0.0)
    faces = [np.array([0.0, one_m, 0.5])] + [np.arange(n + 1) / n for n in nc[:2]]
    hd = h.astype(np.float64)
    pts = []
    for _ in range(n_rand // 3):
        f = np.array([rng.choice(faces[1 + a]) if rng.random() < 0.6 else rng.random()
                      for a in range(2)])
        f = np.where(rng.random(2) < 0.2, rng.choice(faces[0], 2), f)
        pts.append(f @ hd[:2])
    pts = np.array(pts)
    ang = rng.random(len(pts)) * 2 * np.pi
    u = np.stack([np.cos(ang), np.sin(ang), np.zeros_like(ang)], 1)
    scale = r_hi * (1 + rng.choice([-1e-7, -1e-9, 0.0, 1e-9, 1e-7, -0.3], len(pts)))
    partners = pts + u * scale[:, None]
    rand = (rng.random((n_rand - 2 * len(pts), 3)) * 5 - 2) @ hd
    return np.concatenate([pts, partners, rand]).astype(np.float32)


@pytest.mark.parametrize("dims", FLAT_CELLS)
@pytest.mark.parametrize("rel", [0.33, 0.2, 0.05])
def test_single_image_is_the_27_image_minimum_in_the_plane(dims, rel):
    rng = np.random.default_rng(abs(hash((dims, rel))) % 2 ** 32)
    h = _cell(_widened(dims, 2))
    r_hi = rel * _plane_widths(h).min()
    nc, _ = _lib().cells_grid(h, r_hi, 10 ** 12, 2)
    _check_flat(h, r_hi, _adversarial(h, nc, r_hi, 900, rng))


def test_c_just_above_the_cut_off():
    """c_z barely above r_hi + M and a tilted c: the images one c away are just out of
    range and must never be the minimum."""
    rng = np.random.default_rng(3)
    h = np.array([[24, 0, 0], [-12, 20.78461, 0], [7, -5, 100]], np.float32)
    r_hi = 6.0
    _, m = _lib().cells_grid(h, r_hi, 10 ** 12, 2)      # M does not depend on c
    h[2, 2] = np.nextafter(np.float32(r_hi + m), np.float32(np.inf))
    nc, m2 = _lib().cells_grid(h, r_hi, 10 ** 12, 2)
    assert m2 == m and h[2, 2] >= r_hi + m
    h_low = h.copy()
    h_low[2, 2] = np.float32(r_hi)
    with pytest.raises(ValueError, match="c_z"):
        _lib().cells_grid(h_low, r_hi, 10 ** 12, 2)
    _check_flat(h, r_hi, _adversarial(h, nc, r_hi, 900, rng))


def test_large_flat_cell_where_float32_rounding_of_dx_matters():
    rng = np.random.default_rng(7)
    h = _cell(_widened((150.0, 150.0, 40.0, 90.0, 90.0, 120.0), 2))
    r_hi = 1.0
    nc, margin = _lib().cells_grid(h, r_hi, 10 ** 12, 2)
    assert min(nc[:2]) >= 100 and margin > 1e-5 * r_hi
    _check_flat(h, r_hi, _adversarial(h, nc, r_hi, 900, rng))
