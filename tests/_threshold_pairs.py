"""Pairs whose reference squared distance straddles the RDF thresholds as tightly as float32
inputs allow, the reference d2 they are judged by, and the error model of the branch-free
bin guess (rdf_device.cuh::slot_fast_parts).

Used by test_host_bin_lookup.py (CPU) and test_gpu_bin_lookup.py (GPU).

Generator: for a threshold T[k] = min{x : sqrt(x) >= edge_k} a centre c and a partner
p ~ c + sqrt(T[k]) u are placed, then coordinate a = argmax |u_a| is stepped through its
float32 neighbours (of the partner, or of the centre where that one is larger).  Along that walk the reference d2 is monotone, so of
the candidates the one with the largest d2 below T[k] and the one with the smallest d2 at
or above it are one float32 step apart: no pair of float32 inputs lies closer to T[k] on
either side along that direction.

Reference d2:
  orthorhombic  _filter_model.ref_d2 of the float32 differences (rdf.cu header);
  triclinic     both coordinates wrapped into the cell (wrap), then the shortest of the 27
                images of the float32 difference (image_d2), as rdf_tri.cu computes it.
"""
import numpy as np

import _filter_model as fm

F32, F64 = np.float32, np.float64
M27 = np.array([(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)])


# ---- reference squared distances ---------------------------------------------------------

def wrap(p, h):
    """tri_wrap_kernel: along c, then b, then a, in double, rounded to float32."""
    ax, bx, by, cx, cy, cz = (float(h[0, 0]), float(h[1, 0]), float(h[1, 1]), float(h[2, 0]),
                              float(h[2, 1]), float(h[2, 2]))
    x, y, z = (p[:, k].astype(F64) for k in range(3))
    s = np.floor(z / cz)
    x, y, z = x - s * cx, y - s * cy, z - s * cz
    s = np.floor(y / by)
    x, y = x - s * bx, y - s * by
    x = x - np.floor(x / ax) * ax
    return np.stack([x, y, z], 1).astype(F32)


def image_d2(dx, h, m):
    """tri_image_d2 with the shift terms h_k * i."""
    h = h.astype(F64)
    ix, iy, iz = (m[..., k].astype(F64) for k in range(3))
    rx = ((dx[..., 0] + h[0, 0] * ix) + h[1, 0] * iy) + h[2, 0] * iz
    ry = (dx[..., 1] + h[1, 1] * iy) + h[2, 1] * iz
    rz = dx[..., 2] + h[2, 2] * iz
    return (rx * rx + ry * ry) + rz * rz


def tri_ref_d2(c, p, h):
    """The reference's d2 of the pairs (c[i], p[i]) in the lower-triangular cell h."""
    dx = (wrap(p, h) - wrap(c, h)).astype(F64)
    return np.min([image_d2(dx, h, np.broadcast_to(m, dx.shape)) for m in M27], axis=0)


def ref_d2(c, p, box):
    """box: [3] orthorhombic edges or a 3x3 lower-triangular cell."""
    box = np.asarray(box, F32)
    if box.ndim == 2:
        return tri_ref_d2(c, p, box)
    return fm.ref_d2((p - c).astype(F32), box)


# ---- the generator -----------------------------------------------------------------------

KINDS = ("axis", "diag", "face")


def _directions(rng, kind, n, drop):
    axes = [a for a in range(3) if a != drop]
    if kind == "diag":
        u = np.zeros((n, 3))
        u[:, axes] = rng.choice([-1.0, 1.0], (n, len(axes))) * rng.uniform(0.5, 1.0,
                                                                         (n, len(axes)))
    else:
        u = np.zeros((n, 3))
        u[np.arange(n), rng.choice(axes, n)] = rng.choice([-1.0, 1.0], n)
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def straddle_pairs(box, thr, ks, rng, kinds=KINDS, reps=1, drop=None, steps=48, grid=None):
    """For every k in ks and kind: the two partners that straddle T[k] (see the module
    docstring).  box: [3] edges or a 3x3 lower-triangular cell; centres lie in the cell.
    "face" puts the displacement across a periodic face (partner on the far side of the
    cell, image shift not zero).  grid: centres on multiples of it (dyadic boxes: the
    partner at exactly sqrt(T[k]) is representable).  Returns (c, p, d2, k, above) with
    float32 [n, 3] coordinates, the reference d2, the threshold index and whether
    d2 >= T[k]; per kind the pairs below come first, then those above, row for row.
    Thresholds no walk brackets (T[0] = 0; an axis at half a box) are left out."""
    box = np.asarray(box, F32)
    tri = box.ndim == 2
    h = box.astype(F64) if tri else np.diag(box.astype(F64))
    ks = np.repeat(np.asarray(ks), reps)
    out = []
    for kind in kinds:
        n = len(ks)
        u = _directions(rng, kind, n, drop)
        dist = np.sqrt(thr[ks])
        disp = u * dist[:, None]
        frac = rng.uniform(0.2, 0.8, (n, 3))
        # "face": the lattice direction along which the displacement moves farthest; the
        # centre next to that face, the partner's image on the near side
        fd = disp @ np.linalg.inv(h)
        lat = np.argmax(np.abs(fd), axis=1)
        s = np.sign(fd[np.arange(n), lat])
        if kind == "face":
            frac[np.arange(n), lat] = np.where(s > 0, 0.995, 0.005)
        if drop is not None:
            frac[:, drop] = 0.0
        c = frac @ h
        if grid is not None:
            c = np.round(c / grid) * grid
        c = c.astype(F32)
        p0 = c.astype(F64) + disp
        if kind == "face":
            p0 -= s[:, None] * h[lat]
        p0 = p0.astype(F32)
        if drop is not None:
            p0[:, drop] = 0.0
        a = np.argmax(np.abs(u), axis=1)
        sides = _straddle(c, p0, a, box, thr[ks], steps)
        ok = np.isfinite(sides[0][2])
        if kind == "face":
            # keep the pairs whose reference image is not the zero one on both sides (the
            # triclinic wrap can undo the crossing)
            for cc, pp, _ in sides:
                ok &= _crosses(cc, pp, box)
        for above, (cc, pp, d2) in enumerate(sides):
            out.append((cc[ok], pp[ok], d2[ok], ks[ok], np.full(ok.sum(), bool(above))))
    cat = lambda i: np.concatenate([o[i] for o in out])
    return cat(0), cat(1), cat(2), cat(3), cat(4)


def _crosses(c, p, box):
    """The reference's minimum image of the pair is not the zero image."""
    if box.ndim == 2:
        dx = (wrap(p, box) - wrap(c, box)).astype(F64)
        return image_d2(dx, box, np.zeros(dx.shape, np.int64)) > tri_ref_d2(c, p, box)
    return (np.abs((p - c).astype(F64)) > box.astype(F64) / 2).any(1)


def _straddle(c, p0, a, box, t, steps):
    """Steps coordinate a of the partner -- of the centre where that one is larger, its ulp
    sets the resolution of the float32 difference -- by -steps..steps float32 neighbours;
    returns ((c, p, d2) below t, (c, p, d2) at or above t), d2 = inf where the walk does
    not cross t."""
    n = len(c)
    rows = np.arange(n)
    move_c = np.abs(c[rows, a]) > np.abs(p0[rows, a])
    base = np.where(move_c, c[rows, a], p0[rows, a])
    cand = [base]
    lo, hi = base.copy(), base.copy()
    for _ in range(steps):
        lo = np.nextafter(lo, F32(-np.inf))
        hi = np.nextafter(hi, F32(np.inf))
        cand += [lo.copy(), hi.copy()]
    best_b = [c.copy(), p0.copy(), np.full(n, -np.inf)]
    best_a = [c.copy(), p0.copy(), np.full(n, np.inf)]
    for v in cand:
        cc, p = c.copy(), p0.copy()
        cc[rows[move_c], a[move_c]] = v[move_c]
        p[rows[~move_c], a[~move_c]] = v[~move_c]
        d2 = ref_d2(cc, p, box)
        for best, sel in ((best_b, (d2 < t) & (d2 > best_b[2])),
                          (best_a, (d2 >= t) & (d2 < best_a[2]))):
            best[0][sel], best[1][sel], best[2][sel] = cc[sel], p[sel], d2[sel]
    # both sides found: adjacent walk positions bracket t
    found = np.isfinite(best_b[2]) & np.isfinite(best_a[2])
    for best in (best_b, best_a):
        best[2] = np.where(found, best[2], np.inf)
    return best_b, best_a


def threshold_sample(n_bins, rng, n_max=40):
    """T[0], T[1], T[n_bins - 1], T[n_bins] and a random selection of the others."""
    keep = {0, 1, max(0, n_bins - 1), n_bins}
    if n_bins + 1 <= n_max:
        return np.arange(n_bins + 1)
    keep |= set(rng.choice(n_bins + 1, n_max - len(keep), replace=False).tolist())
    return np.array(sorted(keep))


# ---- the bin guess ------------------------------------------------------------------------

HI_MIN, HI_MAX = 0x38000000, 0x47E00000
N_CLASSES = (HI_MAX - HI_MIN + 1) * 8


def guess_float_bits(d2):
    """slot_fast_parts' float32 bits of d2 (numpy restatement of the clamp and the funnel
    shift): uint32."""
    b = np.asarray(d2, F64).view(np.uint64)
    hi = np.clip((b >> np.uint64(32)).astype(np.uint64), HI_MIN, HI_MAX)
    lo = b & np.uint64(0xFFFFFFFF)
    fs = ((hi << np.uint64(3)) | (lo >> np.uint64(29))) & np.uint64(0xFFFFFFFF)
    return ((fs & np.uint64(0x7FFFFFFF)) ^ np.uint64(0x40000000)).astype(np.uint32)


def guess_class(d2):
    """Index of the class of d2 >= 0 on which the guess is constant (rdf_guess_audit_kernel):
    8 * (clamped hi word - HI_MIN) + (lo >> 29)."""
    b = np.asarray(d2, F64).view(np.uint64)
    hi = np.clip((b >> np.uint64(32)).astype(np.int64), HI_MIN, HI_MAX)
    t = ((b & np.uint64(0xFFFFFFFF)) >> np.uint64(29)).astype(np.int64)
    return 8 * (hi - HI_MIN) + t


def class_ends(c):
    """Bit patterns of the smallest and the largest d2 of class c, as the audit kernel
    checks them (the end classes extended to 0 and to the largest finite double)."""
    c = np.asarray(c, np.int64)
    hi = (HI_MIN + (c >> 3)).astype(np.uint64)
    t = (c & 7).astype(np.uint64) << np.uint64(29)
    hi_min = np.where(hi == HI_MIN, np.uint64(0), hi)
    hi_max = np.where(hi == HI_MAX, np.uint64(0x7FEFFFFF), hi)
    return ((hi_min << np.uint64(32)) | t,
            (hi_max << np.uint64(32)) | t | np.uint64(0x1FFFFFFF))


def guess_params(n_bins, r_lo, r_hi):
    """rdf.cu::rdf_bin_guess: (scale, offset) as float32, the exact scale, offset and the
    margin."""
    scale = n_bins / (r_hi - r_lo)
    margin = 1.0 / 64 + n_bins / 524288.0
    off = -r_lo * scale + 0.5 - margin
    return F32(scale), F32(off), scale, off, margin


def guess_error_bound(n_bins, r_lo, r_hi, sqrt_err=2.0 ** -22):
    """(up, down, margin): bounds, in bins, on how far the guess's estimate of
    (sqrt(d2) - r_lo) * scale + 0.5 - margin can lie above / below its exact value for
    sqrt(d2) <= r_hi.  The guess is right for every d2 when up < margin and
    down < 1 - margin.  Terms: sqrt.approx (relative error sqrt_err), the truncation of d2 to
    float32 (down only, relative 2^-23 in d2), the float32 roundings of scale and offset
    and the rounding of the fma (half an ulp of a result below n_bins + 2)."""
    sf, of, scale, off, margin = guess_params(n_bins, r_lo, r_hi)
    sf, of = float(sf), float(of)
    fma = (n_bins + 2) * 2.0 ** -23
    up = r_hi * sf * sqrt_err + max(0.0, r_hi * (sf - scale)) + max(0.0, of - off) + fma
    down = (r_hi * sf * (sqrt_err + 2.0 ** -24) + max(0.0, r_hi * (scale - sf)) +
            max(0.0, off - of) + fma)
    return up, down, margin


# (r_lo, r_hi, n_bins) of the GPU audit sweep: r_lo = 0, then the transition zone where the
# bound above passes the margin (from (99, 100) at 1000 bins), to far past it
SWEEP = ([(0.0, 15.0, 1), (0.0, 15.0, 201), (0.0, 6.0, 4965), (0.0, 8.0, 64)] +
         [(r - 1.0, r, n) for r in (50.0, 100.0, 200.0, 300.0, 500.0, 1000.0)
          for n in (100, 1000, 2000, 4965)] +
         [(9.0, 10.0, 1000), (19.0, 20.0, 1000)])
