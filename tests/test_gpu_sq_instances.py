"""GPU: every compiled instance of the S(q) lattice kernels against the extended-precision
direct sum of ``_sq_reference`` under its worst-case bound.

Each wavevector set here is built to run one chosen instance (``test_host_sq_instances``
checks that through the planner): the 14 ``sq_mma_consume<NT0, NT1>`` of the DMMA kernel, a
mixed multi-block set, the 8 ``R`` of ``sq_lattice_kernel<T>`` for T = double and float, the
table-size limits and deep recurrences.  rho of each group (last frame) and the raw S(q)
accumulator of the pairs (0, 0), (0, 1), (1, 1) over two frames are compared, with
``sort=False``-style raw order (the Context API directly).  Then the chain stride of the
single-chain mode (70,000 chains) and the incoherent ISF over two virtual-frame batches.
"""
import numpy as np
import pytest

import _sq_reference as R

pytestmark = pytest.mark.gpu

PAIRS = [(0, 0), (0, 1), (1, 1)]


def _ctx():
    from mdhelper_b200 import _lib
    return _lib.Context(0)


def _run(kernel, n, b, pos, *, expect=None, f64=False):
    """Configures the raw Context with lattice wavevectors n * b, accumulates ``pos``
    ([F, N, 3]) and returns (kernel run, S raw [3, n_q], rho of the last frame [2, n_q])."""
    ctx = _ctx()
    _, goff = R.group_slices()
    wv = n * b
    ctx.sq_configure(R.N_TOTAL, goff, wv, PAIRS, lattice_n=n, lattice_b=b, mode=kernel)
    ran = ctx.sq_kernel()
    assert ran == (expect or kernel)
    ctx.sq_accumulate(np.ascontiguousarray(pos), 3 * R.N_TOTAL, len(pos), f64=f64)
    S, rho = ctx.sq_fetch(), ctx.sq_fetch_rho()
    ctx.close()
    return ran, S, rho


_REF = {}


def _expected(key, pos, n, b, kernel, coord_rel=0.0):
    k = (key, kernel, coord_rel)
    if k not in _REF:
        _REF[k] = R.expected_s(pos, n, b, kernel, coord_rel)
    return _REF[k]


def _check(key, kernel, n, b, pos, *, expect=None, f64=False, coord_rel=0.0):
    ran, S, rho = _run(kernel, n, b, pos, expect=expect, f64=f64)
    Sr, dS, r, d, margin = _expected(key, pos, n, b, ran, coord_rel)
    assert margin > 1000, margin
    for g in range(2):
        err = np.abs(rho[g] - r[g].astype(np.complex128))
        assert (err <= d[g]).all(), (ran, g, (err / d[g]).max())
    err = np.abs(S - Sr)
    assert (err <= dS).all(), (ran, (err / dS).max())
    return ran, err, dS, Sr


@pytest.fixture(scope="module")
def frames():
    return R.particles()


@pytest.mark.parametrize("inst", R.DMMA_INSTANCES, ids=lambda t: f"{t[0]}{t[1]}")
@pytest.mark.parametrize("kernel", ["lattice_dmma", "lattice_fp64", "general_fp64"])
def test_dmma_instance_sets(frames, inst, kernel):
    pos, b = frames
    n = R.dmma_instance(*inst)
    _check(("inst",) + inst, kernel, n, b, pos)


@pytest.mark.parametrize("kernel", ["lattice_dmma", "lattice_fp64", "general_fp64"])
def test_dmma_mixed_multi_block_set(frames, kernel):
    pos, b = frames
    _check(("mixed",), kernel, R.dmma_mixed(), b, pos)


@pytest.mark.parametrize("second", [False, True], ids=["R", "8+R"])
@pytest.mark.parametrize("R_", range(1, 9))
@pytest.mark.parametrize("kernel", ["lattice_fp64", "lattice_fp32"])
def test_scalar_R(frames, kernel, R_, second):
    pos, b = frames
    n = R.scalar_instance(R_, second)
    ran, err, dS, Sr = _check(("scalar", R_, second), kernel, n, b, pos)
    if kernel == "lattice_fp32":
        rel = err / np.abs(Sr)
        print(f"fp32 R={R_}: max rel err of S {rel.max():.2e}, "
              f"max bound / S {(dS / np.abs(Sr)).max():.2e}")


def test_table_limits(frames):
    from mdhelper_b200 import _lib
    pos, b = frames
    # DMMA tables up to 200 KB: nmax 47 fits, 48 runs the scalar fp64 kernel
    _check(("lim", 47), "lattice_dmma", R.limit_set(47, 47, 47), b, pos)
    _check(("lim", 48), "lattice_dmma", R.limit_set(48, 48, 48), b, pos, expect="lattice_fp64")
    # scalar fp64 tables up to 227 KB: nmax 72 fits, 73 goes to the general kernel under
    # AUTO and is refused for an explicit lattice kernel
    _check(("lim", 72), "lattice_fp64", R.limit_set(72, 72, 72), b, pos)
    _check(("lim", 73), "auto", R.limit_set(73, 73, 73), b, pos, expect="general_fp64")
    n73 = R.limit_set(73, 73, 73)
    for kernel in ("lattice_fp64", "lattice_dmma"):
        ctx = _ctx()
        with pytest.raises(ValueError):
            ctx.sq_configure(R.N_TOTAL, R.group_slices()[1], n73 * b, PAIRS, lattice_n=n73,
                             lattice_b=b, mode=kernel)
        ctx.close()
    assert _lib.sq_plan(R.limit_set(47, 47, 47))["smem_bytes"] <= 200 * 1024


def test_deep_recurrences(frames):
    pos, b = frames
    # 37 steps of E(n + 4) = E(n) E(4) on the DMMA kernel, 200 of E(n + 1) = E(n) E(1) on
    # the scalar one (its tables do not fit the DMMA kernel: lattice_dmma runs it too)
    _check(("deep", 150, 7), "lattice_dmma", R.deep_set(150, 7), b, pos)
    _check(("deep", 150, 7), "lattice_fp64", R.deep_set(150, 7), b, pos)
    _check(("deep", 200, 0), "lattice_fp64", R.deep_set(200, 0), b, pos)
    _check(("deep", 200, 0), "lattice_dmma", R.deep_set(200, 0), b, pos, expect="lattice_fp64")


@pytest.mark.parametrize("kernel", ["lattice_dmma", "lattice_fp64"])
def test_deep_recurrences_float64_far_from_the_origin(kernel):
    """Through mdh_sq_accumulate_f64 with |r| ~ 10^3: the hi + remainder coordinates."""
    pos, b = R.particles(seed=7, offset=1000.0, dtype=np.float64)
    _check(("deep64",), kernel, R.deep_set(150, 7), b, pos, f64=True,
           coord_rel=R.COORD_REL_F64)


# ---- single-chain mode: more chains than one grid dimension -----------------------------

@pytest.mark.parametrize("kernel", ["lattice_dmma", "lattice_fp64"])
def test_scsf_70000_chains(kernel):
    """70,000 chains x 3 monomers: the scalar kernel's grid.y stops at 65,535 and its blocks
    stride over the remaining chains; the DMMA kernel strides over work units."""
    C, M = 70_000, 3
    rng = np.random.default_rng(3)
    L = 40.0
    pos = (rng.random((C * M, 3)) * L).astype(np.float32)
    b = np.full(3, 2 * np.pi / L)
    n = np.array([(x, y, z) for x in range(3) for y in range(3) for z in range(4)],
                 dtype=np.int32)
    ctx = _ctx()
    ctx.sq_configure(C * M, [0, C * M], n * b, [(-1, -1)], lattice_n=n, lattice_b=b,
                     mode=kernel)
    ctx.sq_configure_chains(C, M)
    assert ctx.sq_kernel() == kernel
    ctx.sq_accumulate(pos, 3 * C * M, 1)
    got = ctx.sq_fetch()[0]
    ctx.close()
    chains = pos.reshape(C, M, 3)
    want = np.zeros(len(n))
    bound = np.zeros(len(n))
    for c0 in range(0, C, 10_000):
        part = chains[c0:c0 + 10_000]
        rho = _chain_rho(part, n, b)
        d = R.rho_bound(kernel, part, n, b)
        want += (np.abs(rho) ** 2).astype(np.float64).sum(axis=0)
        bound += R.s_bound(rho, d).sum(axis=0)
    bound += 2 * R.U * C * want                       # fp64 atomics over the chains
    assert (np.abs(got - want) <= bound).all(), (np.abs(got - want) / bound).max()


def _chain_rho(chains, n, b):
    """rho of every chain ([C, M, 3]) in longdouble: [C, n_q]."""
    C, M, _ = chains.shape
    out = np.zeros((C, len(n)), dtype=np.clongdouble)
    c = b.astype(R.LD) / R.TWO_PI
    x = chains.astype(R.LD)
    for m in range(M):
        t = (x[:, m, 0:1] * n[:, 0]) * c[0] + (x[:, m, 1:2] * n[:, 1]) * c[1] \
            + (x[:, m, 2:3] * n[:, 2]) * c[2]
        ph = R.TWO_PI * (t - np.floor(t))
        out += np.cos(ph) + 1j * np.sin(ph)
    return out


# ---- ISF: incoherent part over several virtual-frame batches ----------------------------

@pytest.mark.parametrize("f64", [False, True], ids=["float32", "float64"])
def test_isf_incoherent_over_two_batches(f64):
    """n_points = 32 without q_max: 32,768 wavevectors, so one batch holds 512 virtual
    (frame, lag) frames; 50 frames x 16 lags in one call are 680 of them, two batches.
    Against the same run one frame per call (every call one batch) and, on 100 random
    wavevectors, against the extended-precision sum over the displacements."""
    F, N, n_lags, L = 50, 256, 16, 9.0
    rng = np.random.default_rng(11)
    pos = rng.random((1, N, 3)) * L + rng.normal(0, 0.2, (F, N, 3)).cumsum(axis=0)
    pos = pos.astype(np.float64 if f64 else np.float32)
    idx = np.arange(32)
    n = np.stack(np.meshgrid(idx, idx, idx, indexing="ij"), axis=-1).reshape(-1, 3)
    n = n.astype(np.int32)
    b = np.full(3, 2 * np.pi / L)

    def run(per_call):
        ctx = _ctx()
        ctx.sq_configure(N, [0, N], n * b, [(-1, -1)], lattice_n=n, lattice_b=b)
        ctx.isf_configure(n_lags, True, F)
        for f0 in range(0, F, per_call):
            k = min(per_call, F - f0)
            ctx.isf_accumulate(np.ascontiguousarray(pos[f0:f0 + k]), 3 * N, k, f64=f64)
        out = ctx.isf_fetch(), ctx.sq_kernel()
        ctx.close()
        return out

    (cisf, iisf), ran = run(F)
    (cisf1, iisf1), _ = run(1)
    assert ran == "lattice_dmma"
    scale = N * F
    np.testing.assert_allclose(iisf, iisf1, rtol=1e-12, atol=1e-12 * scale)
    np.testing.assert_allclose(cisf, cisf1, rtol=1e-12, atol=1e-12 * N * scale)
    cols = np.sort(rng.choice(len(n), 100, replace=False))
    nc = n[cols]
    x = pos.astype(R.LD)
    coord_rel = R.COORD_REL_F64_DISP if f64 else 0.0
    for lag in range(n_lags):
        want = np.zeros(len(cols))
        bound = np.zeros(len(cols))
        for t in range(lag, F):
            d = x[t] - x[t - lag]
            want += R.rho_ref(d, nc, b).real.astype(np.float64)
            bound += R.rho_bound(ran, d.astype(np.float64), nc, b, coord_rel=coord_rel)
        bound += 2 * R.U * F * N                    # fp64 sum over the virtual frames
        err = np.abs(iisf[lag, 0, cols] - want)
        assert (err <= bound).all(), (lag, (err / bound).max())
