"""CPU: the reachable-slot bound of the all-pairs fp32 filter's unclamped body.

rdf_device.cuh::filter_reach bounds the fixed-point bin coordinate that filter_d2<true> +
filter_bin2 can produce for a half-box frame; the host sizes the block histogram with it
(rdf_filter.cu::filter_plan) and a frame runs without the slot clamp only if its own
bound lies below the histogram's slot count.  Here the bound is restated and checked
against a float32 evaluation of the kernel's arithmetic on adversarial differences (0, h,
box and 1.5 box on each axis, each moved by a few ulps), with sqrt.approx taken at the
largest relative error the filter accepts, rounded up.
"""
import math

import numpy as np
import pytest

E23, E24 = 2.0 ** -23, 2.0 ** -24
SQRT_ERR = 2.0 ** -22          # rdf_filter_configure declines a larger measured error


def mbound(D, h):
    """filter_halfbox_mbound: bound on the computed |m| of the half-box form."""
    return min(D + h * E23, h) * (1.0 + E23)


def reach(mb, fscale, c0, k, sqrt_err=SQRT_ERR):
    """filter_reach: upper bound of the bin coordinate, in bins relative to slot 0."""
    d2 = (mb[0] ** 2 + mb[1] ** 2 + mb[2] ** 2) * (1.0 + 4.0 * E24)
    s = math.sqrt(d2) * (1.0 + sqrt_err)
    return (s * fscale + c0) * (1.0 + 1e-12) + 2.0 ** -(k + 1)


def f32(x):
    return np.float32(x)


def fma32(a, b, c):
    """float32 fma: the product of two float32 values is exact in float64."""
    return f32(np.float64(a) * np.float64(b) + np.float64(c))


def kernel_coord(df, box, fscale, offm, k, sqrt_err=SQRT_ERR):
    """Bin coordinate (bins above slot 0) of one pair, float32 as in the kernel."""
    m = []
    for d, b in zip(df, box):
        h = f32(b) * f32(0.5)
        e = f32(abs(f32(d)) - h)
        m.append(f32(abs(e) - h))
    d2 = fma32(m[2], m[2], fma32(m[1], m[1], f32(m[0] * m[0])))
    # sqrt.approx at its largest error, upwards, then rounded up to float32
    s = np.nextafter(f32(math.sqrt(float(d2)) * (1.0 + sqrt_err)), f32(np.inf))
    u = fma32(s, fscale, offm)
    return float(u) - 1.5 * 2.0 ** (23 - k)


def layout(n_bins, r_lo, r_hi, box, drop_axis=-1):
    """filter_plan for one frame: (lo, hslots, k, offbase, fscale)."""
    scale = n_bins / (r_hi - r_lo)
    fscale = float(f32(scale))
    lo = math.ceil(r_lo * scale)

    def top(k):
        mb = [mbound(0.0 if a == drop_axis else 0.5 * float(b), 0.5 * float(b))
              for a, b in enumerate(box)]
        c0 = 1.0 + lo - r_lo * scale + 1.0 / 16 + 2.0 ** -(k + 1)
        return math.floor(reach(mb, fscale, c0, k))
    hslots = max(top(9) + 1, n_bins + lo + 2)
    lg = max(hslots - 1, 1).bit_length()
    k = min(16, 22 - lg)
    two_k = 2.0 ** k
    offbase = 1.5 * 2.0 ** (23 - k) + round((1.0 + lo - r_lo * scale) * two_k) / two_k
    return lo, hslots, k, offbase, fscale


def adversarial(box, rng, n=400):
    """Per axis one of 0, +-h, +-box, +-1.5 box, moved by up to 4 ulps."""
    out = []
    for _ in range(n):
        df = []
        for b in box:
            b = f32(b)
            base = f32(rng.choice([0.0, 0.5, -0.5, 1.0, -1.0, 1.5, -1.5]) * float(b))
            for _ in range(int(rng.integers(0, 5))):
                base = np.nextafter(base, f32(np.inf) if rng.random() < 0.5 else f32(-np.inf))
            if abs(float(base)) > 1.5 * float(b):
                base = f32(math.copysign(1.5 * float(b), float(base)))
            df.append(base)
        out.append(df)
    # the corner itself, exactly: d = ||h||
    out.append([f32(0.5) * f32(b) for b in box])
    out.append([f32(1.5) * f32(b) for b in box])
    return out


CASES = [
    # (box, n_bins, range): the benchmark's cfg2 first
    ((29.24, 29.24, 29.24), 201, (0.0, 14.5)),
    ((10.75, 11.5, 12.25), 100, (1.0, 4.5)),
    ((10.75, 11.5, 12.25), 37, (2.25, 2.75)),
    ((12.0, 12.0, 12.0), 1000, (0.0, 6.0)),
    ((3.3333333, 1.0, 7.5), 64, (0.0, 0.5)),
    ((400.0, 380.0, 390.0), 300, (0.0, 4.5)),
]


@pytest.mark.parametrize("box,n_bins,rng_", CASES)
def test_reach_bounds_the_float32_coordinate(box, n_bins, rng_):
    rng = np.random.default_rng(n_bins)
    lo, hslots, k, offbase, fscale = layout(n_bins, *rng_, box)
    # the kernel's offset with the largest window the filter allows (m < 2^k / 16)
    m = 2 ** k // 16 - 1
    offm = f32(offbase + m / 2.0 ** k)
    assert float(offm) == offbase + m / 2.0 ** k
    c0 = float(offm) - 1.5 * 2.0 ** (23 - k)
    mb = [mbound(0.5 * b, 0.5 * b) for b in box]
    bound = reach(mb, fscale, c0, k)
    assert bound < hslots
    worst = 0.0
    for df in adversarial(box, rng):
        u = kernel_coord(df, box, fscale, offm, k)
        assert 0.0 <= u <= bound, (df, u, bound)
        worst = max(worst, u)
    # the bound is tight to well within one slot
    assert bound - worst < 0.5


def test_config2_layout():
    """cfg2: the corner distance ||h|| = 25.3 reaches slot 352; the histogram has 353
    slots x 32 columns (45 KB), k drops from 14 to 13 and two blocks still fit an SM."""
    lo, hslots, k, _, _ = layout(201, 0.0, 14.5, (29.24, 29.24, 29.24))
    assert (lo, hslots, k) == (0, 353, 13)
    hist = hslots * 32 * 4
    smem = hist + 202 * 8 + 2 * (1024 + 4) * 16 + (3072 + 4) * 4
    assert hist < 46 * 1024 and smem < 224 * 1024 // 2 - 1024


def test_lower_limit_shift_keeps_the_coordinate_non_negative():
    """r_lo > 0: the offset is shifted by ceil(r_lo * scale) slots, so a distance of 0
    (and anything below r_lo) lands in a scratch slot at or above 0."""
    for n_bins, r_lo, r_hi in [(100, 1.0, 4.5), (37, 2.25, 2.75), (50, 5.0, 9.0),
                               (7, 0.3, 1.0)]:
        lo, hslots, k, offbase, fscale = layout(n_bins, r_lo, r_hi, (12.0, 12.0, 12.0))
        u0 = kernel_coord([0.0, 0.0, 0.0], (12.0, 12.0, 12.0), fscale, f32(offbase), k)
        assert 0.0 < u0 < lo + 1
        # r_lo itself is the first counted slot, lo + 1
        u = kernel_coord([r_lo, 0.0, 0.0], (12.0, 12.0, 12.0), fscale, f32(offbase), k)
        assert abs(u - (lo + 1)) < 1e-3


def test_dropped_axis_does_not_count():
    """A dropped axis has df = 0, so its edge does not size the histogram."""
    _, h3, _, _, _ = layout(100, 0.0, 5.0, (10.0, 10.0, 1000.0))
    _, h2, _, _, _ = layout(100, 0.0, 5.0, (10.0, 10.0, 1000.0), drop_axis=2)
    assert h2 < 160 < h3
