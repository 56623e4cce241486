"""Bit-level numpy model of the fp32 RDF filter's per-pair arithmetic, the exact fp64
reference it is checked against, and a generator of pairs at bin edges.

Used by test_host_filter_window.py (CPU) and test_gpu_rdf_filter_edges.py (GPU).  The
layout and the per-frame window always come from the library (mdh_rdf_filter_window,
mdhelper_b200._lib.filter_window), never from a Python copy of the formulas.

Model (rdf_device.cuh):
  filter_d2   df = x_j - x_i (float32); half-box form m = ||df| - h| - h with h = box/2,
              rint form r = fma(df, inv, 1.5*2^23) - 1.5*2^23, m = fma(-box, r, df);
              d2 = fma(mz, mz, fma(my, my, mx*mx)).  Every fma is correctly rounded
              (TwoSum of the exact double product and the addend, ties fixed by the error
              term), so there is no double rounding.
  filter_bin2 s = sqrt.approx.ftz(d2): d2 below 2^-126 flushes to 0; otherwise s is any
              float32 in [sqrt(d2)(1 - sqrt_err), sqrt(d2)(1 + sqrt_err)] -- the model takes
              both extremes; u = bits(fma(s, scale, offm)) (- cbits when LOWER).
  words       all-pairs: t = u >> (k - cb - 2), clamped bodies t = min(t, tmax), slot =
              (t & tmask) >> (cb + 2); cell list: w = min(u >> (k - sb), span_l >> (k - sb)),
              slot = (w - base) >> sb.
Reference (rdf.cu header): s = inv*df, r = (s + 1.5*2^52) - 1.5*2^52, m = box*(s - r),
d2 = (mx*mx + my*my) + mz*mz in fp64, binned with _binning.squared_thresholds.
"""
import numpy as np

F32, F64 = np.float32, np.float64
MAGIC32 = F32(12582912.0)            # 1.5 * 2^23
MAGIC64 = 6755399441055744.0         # 1.5 * 2^52
E24 = 2.0 ** -24


# ---- float32 arithmetic -------------------------------------------------------------

def _rn32(s, t):
    """float32 nearest of the exact value s + t (s a double, |t| <= ulp(s) / 2)."""
    r = s.astype(F32)
    rd = r.astype(F64)
    o = np.nextafter(r, np.where(s > rd, F32(np.inf), F32(-np.inf)).astype(F32))
    od = o.astype(F64)
    tie = (s == 0.5 * (rd + od)) & (t != 0)
    pick_o = tie & ((t > 0) == (od > rd))
    return np.where(pick_o, o, r).astype(F32)


def fma32(a, b, c):
    """Correctly rounded float32 fma(a, b, c): the product of two float32 values is exact in
    double, the sum is TwoSum-split into s + t and rounded once."""
    a, b, c = np.broadcast_arrays(np.asarray(a, F32), np.asarray(b, F32), np.asarray(c, F32))
    p = a.astype(F64) * b.astype(F64)
    c64 = c.astype(F64)
    s = p + c64
    bb = s - p
    t = (p - (s - bb)) + (c64 - bb)
    return _rn32(s, t)


def _ceil32(x):
    r = x.astype(F32)
    return np.where(r.astype(F64) < x, np.nextafter(r, F32(np.inf)), r).astype(F32)


def _floor32(x):
    r = x.astype(F32)
    return np.where(r.astype(F64) > x, np.nextafter(r, F32(-np.inf)), r).astype(F32)


def filter_d2(df, box, half):
    """filter_d2<HALF>: df float32 [n, 3] (the reference's own differences), box [3]."""
    box = np.asarray(box, F32)
    m = np.empty_like(df)
    for k in range(3):
        d = df[:, k]
        if half:
            nh = F32(-0.5) * box[k]                       # exact
            m[:, k] = np.abs(np.abs(d) + nh) + nh
        else:
            inv = F32(1.0 / float(box[k]))
            r = fma32(d, inv, MAGIC32) - MAGIC32           # exact subtraction
            m[:, k] = fma32(-box[k], r, d)
    return fma32(m[:, 2], m[:, 2], fma32(m[:, 1], m[:, 1], m[:, 0] * m[:, 0]))


def filter_coords(d2, fscale, offm, sqrt_err):
    """filter_bin2 before the LOWER subtraction: the float32 bit patterns of fma(s, scale,
    offm) for the two extremes of sqrt.approx.ftz, as int64 [2, n]."""
    d2 = np.where(d2 < F32(2.0 ** -126), F32(0.0), d2)  # ftz
    t = np.sqrt(d2.astype(F64))
    out = []
    for s in (_ceil32(t * (1.0 - sqrt_err)), _floor32(t * (1.0 + sqrt_err))):
        e = fma32(s, F32(fscale), F32(offm))
        out.append(e.view(np.uint32).astype(np.int64))
    return np.stack(out)


# ---- exact reference ---------------------------------------------------------------

def ref_d2(df, box):
    """The reference's fp64 squared minimum-image distance of float32 differences."""
    box64 = np.asarray(box, F32).astype(F64)
    inv = (1.0 / box64).astype(F32).astype(F64)
    d = df.astype(F64)
    s = inv * d
    r = (s + MAGIC64) - MAGIC64
    m = box64 * (s - r)
    return (m[:, 0] * m[:, 0] + m[:, 1] * m[:, 1]) + m[:, 2] * m[:, 2]


def ref_slots(d2, thr):
    """slot = bin + 1; 0 below the range, n_bins + 1 at or above its end."""
    return np.searchsorted(thr, d2, side="right")


# ---- the kernels' word addressing ---------------------------------------------------

def allpairs_slot(u, L, clamp):
    """The histogram slot a pair of the all-pairs kernel is added to (u with cbits removed
    when LOWER, as filter_bin2 returns it)."""
    k, cb, lg, hs = L["k"], L["cb"], L["lg"], L["hslots"]
    tshift = k - cb - 2
    low = (4 << cb) - 1
    tmask = ((4 << (cb + lg)) - 1) & ~low
    tmax = ((((0 if L["lower"] else L["cbits"]) >> k) + hs - 1) << (cb + 2)) | low
    t = u >> tshift
    if clamp:
        t = np.minimum(t, tmax)
    return (t & tmask) >> (cb + 2)


def cell_slot(u, L, sb):
    """The slot of the cell-pair kernel's word for 2^sb sub-bins per bin."""
    shift = L["k"] - sb
    span_l = L["span"] if L["lower"] else L["cbits"] + L["span"]
    base = 0 if L["lower"] else L["cbits"] >> shift
    w = np.minimum(u >> shift, span_l >> shift)
    return (w - base) >> sb


def uncertain(u, L, wlim):
    span_l = L["span"] if L["lower"] else L["cbits"] + L["span"]
    return (u < span_l) & ((u & ((1 << L["k"]) - 1)) < wlim)


def lowered(bits, L):
    """filter_bin2's u: the bits, minus cbits when LOWER (modulo 2^32)."""
    return (bits - L["cbits"]) % (1 << 32) if L["lower"] else bits


# ---- pairs at bin edges ---------------------------------------------------------------

def extents(c, p):
    """float32 {min x, y, z, max x, y, z} of both groups, as the pack kernel reduces them."""
    return (np.concatenate([c.min(0), c.max(0)]).astype(F32),
            np.concatenate([p.min(0), p.max(0)]).astype(F32))


def edge_sample(n_bins, r_lo, r_hi, rng, n_max=48):
    """Bin edges to probe: all of them for few bins, else r_lo, the first two, the last two,
    r_hi and a random selection."""
    idx = np.arange(n_bins + 1)
    if n_bins + 1 > n_max:
        keep = {0, 1, 2, n_bins - 1, n_bins}
        keep |= set(rng.choice(n_bins + 1, n_max - len(keep), replace=False).tolist())
        idx = np.array(sorted(keep))
    return r_lo + idx * ((r_hi - r_lo) / n_bins)


T_SWEEP = np.array([0.0, 0.25, -0.25, 0.5, -0.5, 1.0, -1.0, 1.5, -1.5, 2.0, -2.0, 3.0, -3.0,
                    4.0, -4.0])


def _unit(rng, n, drop):
    u = rng.normal(size=(n, 3))
    if drop is not None:
        u[:, drop] = 0
    return u / np.linalg.norm(u, axis=1, keepdims=True)


def edge_pairs(rng, box, edges, w, kinds, region, drop=None, reps=1, n_shift=0):
    """Pairs (c, p) of float32 coordinates whose minimum-image distance is about e + t w for
    every edge e and t in T_SWEEP (w: the frame's window half-width in distance units).
    Every coordinate lies in [0, region_k); candidates that do not fit are dropped.

    kinds: "inside"  random directions, |df_k| < h_k
           "axis"    along one axis
           "h"       one component at +-h_k (the minimum-image switch), moved by a few ulps
           "box"     one axis wrapped: df_k = disp_k -+ box_k (|df| near box)
           "1.5box"  one axis at +-(box_k + h_k): |df| near 1.5 box
           "unwrap"  every axis shifted by up to n_shift boxes (rint form)
           "d2"      along x with small y, z chosen so that the float32 sum of squares
                     rounds as far as it can, both ways
    """
    box = np.asarray(box, F64)
    h = box / 2
    d = (edges[:, None] + T_SWEEP[None, :] * w).ravel()
    d = np.repeat(d[d >= 0], reps)
    axes = [a for a in range(3) if a != drop]
    out = []
    for kind in kinds:
        n = len(d)
        if kind == "d2":
            out.append(_d2_probe(rng, d, box, region, drop))
            continue
        if kind == "axis":
            disp = np.zeros((n, 3))
            ax = rng.choice(axes, n)
            disp[np.arange(n), ax] = d * rng.choice([-1.0, 1.0], n)
        elif kind in ("h", "1.5box"):
            ax = rng.choice(axes, n)
            hk = h[ax] * (1 + rng.integers(-4, 5, n) * 2.0 ** -23)
            rest = np.sqrt(np.maximum(d * d - hk * hk, 0.0))
            disp = _unit(rng, n, drop) * rest[:, None]
            disp[np.arange(n), ax] = hk * rng.choice([-1.0, 1.0], n)
            ok = d >= hk
            disp = disp[ok]
            ax = ax[ok]
        else:
            disp = _unit(rng, n, drop) * d[:, None]
        df = disp.copy()
        if kind in ("box", "1.5box"):
            if kind == "box":
                ax = rng.choice(axes, len(df))
            sgn = np.sign(df[np.arange(len(df)), ax])
            sgn[sgn == 0] = 1.0
            df[np.arange(len(df)), ax] -= sgn * box[ax]
        elif kind == "unwrap":
            shift = rng.integers(-n_shift, n_shift + 1, size=df.shape)
            if drop is not None:
                shift[:, drop] = 0
            df += shift * box
        if kind not in ("box", "1.5box", "unwrap"):
            ok = np.all(np.abs(disp) < h, axis=1)
            df = df[ok]
        out.append(_place(rng, df, region, drop))
    c = np.concatenate([o[0] for o in out])
    p = np.concatenate([o[1] for o in out])
    return c, p


def _place(rng, df, region, drop):
    """Centres c and partners p = c + df, both inside [0, region)."""
    region = np.asarray(region, F64)
    lo = np.maximum(0.0, -df)
    hi = region - np.maximum(0.0, df)
    ok = np.all(hi > lo, axis=1)
    df, lo, hi = df[ok], lo[ok], hi[ok]
    c = (lo + rng.random(df.shape) * (hi - lo)).astype(F32)
    p = (c.astype(F64) + df).astype(F32)
    if drop is not None:
        c[:, drop] = 0
        p[:, drop] = 0
    return c, p


def _d2_probe(rng, d, box, region, drop, n_cand=24):
    """Along x (or y when x is dropped) with tiny other components: of n_cand candidates per
    target keep the two whose float32 sum of squares has the largest relative error either
    way (the (1 + 2^-24)^3 term of the bound)."""
    ax = 1 if drop == 0 else 0
    others = [a for a in range(3) if a not in (ax, drop)]
    d = d[(d > 0) & (d < box[ax] / 2)]
    n = len(d)
    dd = np.repeat(d, n_cand)
    # half an ulp of d^2: a component whose square is about that makes the fma round
    hulp = np.ldexp(1.0, np.frexp(dd * dd)[1] - 25)
    df = np.zeros((len(dd), 3))
    df[:, ax] = dd * rng.choice([-1.0, 1.0], len(dd))
    for a in others:
        df[:, a] = np.sqrt(hulp * rng.uniform(0.6, 1.6, len(dd))) * rng.choice([-1.0, 1.0],
                                                                              len(dd))
    c, p = _place(rng, df, region, drop)
    dff = p - c
    if len(dff) == 0:
        return c, p
    fp = filter_d2(dff, box.astype(F32), True).astype(F64)
    x = dff.astype(F64)
    ex = (x * x).sum(1)
    rel = np.where(ex > 0, (fp - ex) / np.maximum(ex, 1e-300), 0.0)
    n_keep = len(rel) // n_cand
    rel = rel[:n_keep * n_cand].reshape(n_keep, n_cand)
    base = np.arange(n_keep) * n_cand
    pick = np.concatenate([base + rel.argmax(1), base + rel.argmin(1)])
    return c[pick], p[pick]


def frame_window(L, W):
    """(k, m, magic): fraction bits, window half-width (units of 2^-k) and 1.5 * 2^(23-k)."""
    k = L["k"]
    return k, (W["wlim"] - 1) // 2, 1.5 * 2.0 ** (23 - k)


def window_distance(L, W, scale):
    k, m, _ = frame_window(L, W)
    return m * 2.0 ** -k / scale


def check_pairs(c, p, box, thr, L, W, body, sqrt_err, r_lo, scale, n_bins, sb=0):
    """Runs the model on the pairs of one frame for one body ("unclamped", "clamped" or
    "cells") and returns a dict of findings: wrong certain slots, pairs of an unclamped frame
    outside its histogram, the largest coordinate error and the frame's mu."""
    box = np.asarray(box, F32)
    df = p - c
    half = body != "cells" and W["halfbox"] == 1
    d2f = filter_d2(df, box, half)
    d2r = ref_d2(df, box)
    xs = ref_slots(d2r, thr) + L["lo"]
    k, m, magic = frame_window(L, W)
    bits = filter_coords(d2f, L["scale"], W["offm"], sqrt_err)        # [2, n]
    dmax = (n_bins / scale + r_lo) + 2.0 / scale
    dref = np.sqrt(d2r)
    exact = (dref - r_lo) * scale + 1.0 + L["lo"]
    res = {"wrong": 0, "outside": 0, "err": 0.0, "n": len(df), "uncertain": 0}
    for b in bits:
        u = lowered(b, L)
        unc = uncertain(u, L, W["wlim"])
        res["uncertain"] += int(unc.sum())
        if body == "cells":
            fs = cell_slot(u, L, sb) + L["lo"]
        else:
            fs = allpairs_slot(u, L, clamp=body == "clamped")
        counted = lambda s: (s >= L["lo"] + 1) & (s <= L["lo"] + n_bins)
        bad = ~unc & (fs != xs) & (counted(xs) | counted(fs))
        res["wrong"] += int(bad.sum())
        if body == "unclamped":
            res["outside"] += int(((b - L["cbits"]) >> k >= L["hslots"]).sum() +
                                  (b < L["cbits"]).sum())
        val = np.frombuffer(b.astype(np.uint32).tobytes(), F32).astype(F64)
        model = val - magic - m * 2.0 ** -k
        inr = dref <= dmax
        if inr.any():
            res["err"] = max(res["err"], float(np.abs(model - exact)[inr].max()))
    return res
