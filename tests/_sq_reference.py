"""Extended-precision direct sum of the S(q) kernels and a worst-case bound on their error.

``rho_ref`` is rho(q) = sum_j exp(i q . r_j) for lattice wavevectors q = n * b, evaluated in
``np.longdouble`` (x86-64: 64-bit significand, unit roundoff 2^-64).  ``rho_bound`` bounds
|rho_kernel - rho| per wavevector from what each kernel does (``mdhelper_b200/csrc/sq.cu``);
nothing in it is fitted to observed errors.  ``s_bound`` carries that to |rho|^2 and the
cross terms.  The builders at the end make the wavevector sets whose plans run one chosen
kernel instance; the CPU test checks them through ``mdh_sq_plan_items``, the GPU test runs
them.
"""
import math

import numpy as np

LD = np.longdouble
U = 2.0 ** -53          # fp64 unit roundoff
UF = 2.0 ** -24         # fp32 unit roundoff
CHUNK_MAX = 4096        # particles per chunk of every S(q) kernel (sq_build_chunks)
# coordinate error of the float64 entry points: float32 hi + float32 remainder, added in fp64
# (sq_split_kernel): |x - x~| <= 2^-48 |x| + u |x|; the ISF's float64 window takes the
# displacement in fp64 first (one more u)
COORD_REL_F64 = 2.0 ** -48 + U
COORD_REL_F64_DISP = 2.0 ** -48 + 2 * U


def _two_pi():
    # 2 pi to the longdouble's precision from the float64 split pi = hi + lo
    hi = LD(np.pi)
    lo = LD(1.2246467991473532e-16)            # pi - fl64(pi)
    return 2 * (hi + lo)


TWO_PI = _two_pi()
REF_U = float(np.finfo(LD).eps) / 2             # 2^-64 on x86-64


def rho_ref(pos, lattice_n, lattice_b):
    """rho[q] = sum_j exp(i q_q . r_j), q_q = lattice_n[q] * lattice_b, in longdouble.

    ``pos`` ([N, 3], float32 or float64; pass longdouble for displacements taken exactly)
    is used as given.  The phase is reduced before the sine: t = sum_a n_a x_a (b_a / 2 pi),
    phase = 2 pi frac(t).  n_a x_a is exact (|n| < 2^11, 53-bit x); with (b_a / 2 pi) and
    the two sums rounded, |t~ - t| <= 5 * 2^-64 * T, T = sum_a |n_a b_a x_a| / 2 pi, and
    sinl / cosl add 2^-64 each.  Per particle that is <= 2^-64 (10 pi T + 2), summed over
    N terms pairwise (log2 N roundings of <= N per component): ``ref_error`` returns it.  Every
    kernel's bound has >= 2^-53 |b_a x_a| n_a per term from forming its own argument, so the
    reference's own error stays > 1000x below every tolerance it is used with
    (``tests/test_host_sq_instances.py`` asserts the margin case by case)."""
    x = np.asarray(pos)
    x = x.astype(LD) if x.dtype != LD else x
    n = np.asarray(lattice_n, dtype=np.int64).reshape(-1, 3)
    assert np.abs(n).max() < 2 ** 11
    c = np.asarray(lattice_b, dtype=np.float64).astype(LD) / TWO_PI
    out = np.zeros(len(n), dtype=np.clongdouble)
    step = max(1, 2_000_000 // max(1, len(x)))
    for q0 in range(0, len(n), step):
        nq = n[q0:q0 + step].astype(LD)
        t = (x[:, 0:1] * nq[:, 0]) * c[0] + (x[:, 1:2] * nq[:, 1]) * c[1] \
            + (x[:, 2:3] * nq[:, 2]) * c[2]
        ph = TWO_PI * (t - np.floor(t))
        out[q0:q0 + step] = np.cos(ph).sum(axis=0) + 1j * np.sin(ph).sum(axis=0)
    return out


def ref_error(pos, lattice_n, lattice_b):
    """Bound on |rho_ref - rho| (see ``rho_ref``)."""
    T = _theta(pos, lattice_n, lattice_b) / (2 * math.pi)
    N = len(pos)
    # numpy sums pairwise: <= ceil(log2 N) roundings of <= N per component
    return REF_U * (10 * math.pi * T + 2 * N + 2 * N * (math.ceil(math.log2(max(N, 2))) + 1))


def _theta(pos, lattice_n, lattice_b):
    """sum_j sum_a |n_a b_a x_ja| per wavevector (float64 is plenty for a bound)."""
    X = np.abs(np.asarray(pos, dtype=np.float64)).sum(axis=0)         # [3]
    n = np.asarray(lattice_n, dtype=np.float64).reshape(-1, 3)
    return (n * np.abs(np.asarray(lattice_b, dtype=np.float64)) * X).sum(axis=1)


def rho_bound(kernel, pos, lattice_n, lattice_b, *, coord_rel=0.0, chunk_max=CHUNK_MAX):
    """Worst-case |rho_kernel(q) - rho(q)| of one group (its particles ``pos``) per
    wavevector, for ``kernel`` in lattice_dmma / lattice_fp64 / lattice_fp32 /
    general_fp64.  ``coord_rel``: relative error of the coordinate the kernel reads
    (0 for float32 input and for differences of float32 coordinates, which fp64 forms
    exactly; ``COORD_REL_F64`` / ``COORD_REL_F64_DISP`` for the float64 paths).

    Notation: u = 2^-53, u_f = 2^-24, n = lattice index on one axis, x = coordinate, E(n) =
    exp(i n b x) with |E| = 1; delta = bound on |computed - exact|.  A complex product
    a*b of two values of modulus <= 1 rounds each component at most twice with
    |x1 y1| + |x2 y2| <= |a||b|, so it adds <= 2 sqrt(2) u (1 + u) <= 3u.  Terms of second
    order in u (< 1e-20 relative here) are covered by that rounding-up.

    Phase factors
      lattice_fp64 / fp32 (producer: one sincos, then E(n+1) = E(n) E(1)):
        arg = fl(b x): |arg - b x| <= (u + coord_rel) |b x|; sincos 2 ulp per component
        (CUDA fp64 sin / cos), <= 4 sqrt(2) u = 5.66u in modulus; n steps of the
        recurrence, each passing the factor error on and adding 3u:
            delta E(n) <= n (u + coord_rel) |b x| + n (5.66u + 3u).
      lattice_dmma (producer: sincospi, E(2) = E(1)^2, E(4) = E(2)^2, four interleaved
        recurrences E(n + 4) = E(n) E(4); the second half of E_z starts at
        E(n0) = E(4)^(n0 / 4)):
        th = fl(fl(b * fl(1/pi)) * x): 3u + coord_rel relative; sincospi 2 ulp:
            d1 = (3u + coord_rel) |b x| + 5.66u,  d2 = 2 d1 + 3u,  d4 = 4 d1 + 9u,
            E(1..3) <= 3 d1 + 6u, one more product for the second half's start (+3u),
            floor(n / 4) products by E(4) on the way to entry n (n0 / 4 of them to
            reach n0, the rest after it: floor(n / 4) either way):
            delta E(n) <= floor(n / 4) (d4 + 3u) + 3 d1 + 9u.
      general_fp64: arg = fl(q . x) with q = fl(n b): |arg - q.x| <= (4u + coord_rel) sum_a
        |n_a b_a x_a|; one sincos: + 5.66u.
    Product and sum (m = particles of a chunk <= min(N, 4096), partial sums <= m):
      lattice_fp64: A = E_x E_y (+3u), A E_z accumulated by 2 FMAs per component per
        particle (roundings <= u |partial|): per chunk <= sqrt(2) u m (m + 1).
      lattice_fp32: the same with table entries rounded to float (+u_f each, three per
        term), A in float (+3 u_f) and float accumulators: sqrt(2) u_f m (m + 1) per chunk.
      lattice_dmma: A = E_x E_y (+3u); 3M: P1 = sum A_r B_r, P2 = sum A_i B_i,
        P3 = sum (A_r + A_i)(B_r + B_i), the two sums rounded (+u sqrt(2) each, times
        |other factor| <= sqrt(2): +4u per term on P3).  A DMMA is charged one rounding
        per product and one per addition: terms <= 1 (P1, P2) or <= 2 (P3) give
        |delta P1|, |delta P2| <= u m (m + 3) / 2, |delta P3| <= u m (m + 3); Re = P1 - P2,
        Im = P3 - P1 - P2 carry those absolute errors (the 3M step) plus their own
        roundings (<= u m, 2 u 4m):  per chunk <= u (2 m (m + 3) + 9 m).
      general_fp64: one rounding per particle per component: sqrt(2) u m (m + 1) / 2.
    Chunks are added by fp64 atomics into rho (partial sums <= N, at most N / 32 + 1
    chunks per group): + sqrt(2) u N (N / 32 + 1).
    The particle terms are summed over the group, with the phase parts linear in
    sum_j |x_ja|."""
    pos = np.asarray(pos, dtype=np.float64)
    N = pos.shape[-2]                                      # [..., N, 3]: groups, e.g. chains
    n = np.asarray(lattice_n, dtype=np.float64).reshape(-1, 3)
    b = np.abs(np.asarray(lattice_b, dtype=np.float64))
    bX = (b * np.abs(pos).sum(axis=-2))[..., None, :]     # sum_j |b_a x_ja|, [..., 1, 3]
    m = min(N, chunk_max)
    r2 = math.sqrt(2.0)
    if kernel in ("lattice_fp64", "lattice_fp32"):
        phase = (n * bX).sum(axis=-1) * (U + coord_rel)
        const = N * (n.sum(axis=1) * (5.66 * U + 3 * U) + 3 * U)
        if kernel == "lattice_fp64":
            acc = r2 * U * N * (m + 1)
        else:
            const = const + N * 6 * UF
            acc = r2 * UF * N * (m + 1)
        per = phase + const + acc
    elif kernel == "lattice_dmma":
        fl4 = np.floor(n / 4)
        # the phase part of d1 enters 4 floor(n / 4) + 3 times per axis
        phase = ((4 * fl4 + 3) * bX).sum(axis=-1) * (3 * U + coord_rel)
        d1c = 5.66 * U
        d4c = 4 * d1c + 9 * U
        const = N * ((fl4 * (d4c + 3 * U) + 3 * d1c + 9 * U).sum(axis=1) + 3 * U + 4 * U)
        acc = U * N / m * (2 * m * (m + 3) + 9 * m)
        per = phase + const + acc
    elif kernel == "general_fp64":
        phase = (n * bX).sum(axis=-1) * (4 * U + coord_rel)
        per = phase + N * 5.66 * U + r2 * U * N * (m + 1) / 2
    else:
        raise ValueError(kernel)
    return per + r2 * U * N * (N / 32 + 1)


def s_bound(rho_j, d_j, rho_k=None, d_k=None):
    """Bound on the error of one frame's S(q) term from the rho bounds: |rho_j|^2 (rho_k
    None) or 2 Re(rho_j conj(rho_k)), each formed by the finalize kernel in fp64 (a few
    roundings of the result's size) and added to the accumulator:
        |delta |rho|^2| <= 2 |rho| d + d^2,
        |delta 2 Re(rho_j rho_k*)| <= 2 (|rho_j| d_k + |rho_k| d_j + d_j d_k)."""
    aj = np.abs(rho_j).astype(np.float64)
    if rho_k is None:
        return 2 * aj * d_j + d_j ** 2 + 4 * U * aj ** 2
    ak = np.abs(rho_k).astype(np.float64)
    return 2 * (aj * d_k + ak * d_j + d_j * d_k) + 8 * U * aj * ak


# ---- wavevector sets that select one kernel instance ---------------------------------

def dmma_instance(a, b):
    """One DMMA warp item with (nt0, nt1) = (a, b): 8 columns (x, 0) of height 8a and,
    for b > 0, 8 columns (x, 1) of height 8b."""
    n = [(x, 0, z) for x in range(8) for z in range(8 * a)]
    n += [(x, 1, z) for x in range(8) for z in range(8 * b)]
    return np.array(n, dtype=np.int32)


DMMA_INSTANCES = [(a, b) for a in range(1, 5) for b in range(0, a + 1)]


def dmma_mixed():
    """Columns of random height 1..40 over a 16 x 16 grid: two blocks of 11 consumer warps
    (producers at warps 3 and 7), one padding item, items starting at nz tile 4."""
    rng = np.random.default_rng(2)
    n = []
    for x in range(16):
        for y in range(16):
            h = int(rng.integers(1, 41))
            n += [(x, y, z) for z in range(h)]
    return np.array(n, dtype=np.int32)


def scalar_instance(R, second_segment=False):
    """64 columns (8 x 8) of height R (or 8 + R): one warp of the scalar kernel with
    R z-terms (after a warp with 8 for ``second_segment``)."""
    h = R + (8 if second_segment else 0)
    return np.array([(x, y, z) for x in range(8) for y in range(8) for z in range(h)],
                    dtype=np.int32)


def limit_set(nx, ny, nz):
    """Sparse set whose largest index per axis is (nx, ny, nz): the tables of the lattice
    kernels are sized by it."""
    n = {(nx, 0, 0), (0, ny, 0), (0, 0, nz), (nx, ny, nz), (1, 2, 3), (0, 0, 0),
         (nx // 2, ny // 3, nz // 2), (nx, 1, 1), (1, ny, 1), (1, 1, nz)}
    return np.array(sorted(n), dtype=np.int32)


def deep_set(nx, nz):
    """Anisotropic set reaching (nx, 0, nz): deep recurrences along x (and z)."""
    n = [(x, 0, z) for x in range(0, nx + 1, 3) for z in range(0, nz + 1)]
    n += [(nx, 0, z) for z in range(nz + 1)]
    return np.unique(np.array(n, dtype=np.int32), axis=0)


# ---- particles of the GPU test (the CPU test evaluates the bounds of the same cases) ----

GROUPS = (263, 437)           # two groups of unequal size, both with a partial sub-chunk
N_TOTAL = sum(GROUPS)
BOX = 11.3


def particles(seed=20261020, frames=2, box=BOX, offset=0.0, dtype=np.float32):
    """[frames, N_TOTAL, 3] coordinates in [offset, offset + box) and the lattice b."""
    rng = np.random.default_rng(seed)
    pos = (offset + rng.random((frames, N_TOTAL, 3)) * box).astype(dtype)
    return pos, np.full(3, 2 * np.pi / box)


def group_slices():
    o = np.concatenate(([0], np.cumsum(GROUPS)))
    return [slice(int(o[g]), int(o[g + 1])) for g in range(len(GROUPS))], o


def expected_s(frames, lattice_n, lattice_b, kernel, coord_rel=0.0):
    """Reference and bound of the raw accumulator of the pairs (0, 0), (0, 1), (1, 1) over
    ``frames`` ([F, N_TOTAL, 3]), the reference rho of the last frame per group and its
    bound, and the smallest ratio bound / reference error met on the way."""
    sl, _ = group_slices()
    n_q = len(lattice_n)
    S = np.zeros((3, n_q))
    dS = np.zeros((3, n_q))
    margin = np.inf
    for f in range(len(frames)):
        r, d = [], []
        for s in sl:
            p = frames[f, s]
            r.append(rho_ref(p, lattice_n, lattice_b))
            d.append(rho_bound(kernel, p, lattice_n, lattice_b, coord_rel=coord_rel))
            margin = min(margin, float((d[-1] / ref_error(p, lattice_n, lattice_b)).min()))
        S[0] += np.abs(r[0]).astype(np.float64) ** 2
        S[1] += 2 * (r[0] * r[1].conj()).real.astype(np.float64)
        S[2] += np.abs(r[1]).astype(np.float64) ** 2
        dS[0] += s_bound(r[0], d[0])
        dS[1] += s_bound(r[0], d[0], r[1], d[1])
        dS[2] += s_bound(r[1], d[1])
    # the finalize kernel's fp64 sum over the frames
    dS += 2 * U * len(frames) * (np.abs(S) + dS)
    return S, dS, r, d, margin
