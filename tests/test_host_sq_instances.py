"""CPU: the wavevector sets of ``test_gpu_sq_instances`` reach the kernel instances they are
built for (``mdh_sq_plan_items``), and the error bounds of ``_sq_reference`` are neither
vacuous nor below the reference's own error."""
import numpy as np
import pytest

import _sq_reference as R
from mdhelper_b200 import _lib


def _instances(n):
    it = _lib.sq_plan_items(n)["mma"]
    return {(int(a), int(b)) for a, b, _, pad in it if not pad}


@pytest.mark.parametrize("inst", R.DMMA_INSTANCES, ids=lambda t: f"{t[0]}{t[1]}")
def test_each_dmma_builder_runs_exactly_its_instance(inst):
    n = R.dmma_instance(*inst)
    plan = _lib.sq_plan_items(n)["mma"]
    assert plan.tolist() == [[inst[0], inst[1], 0, 0]]
    assert (_lib.sq_plan(n)["coverage"] == 1).all()


def test_builders_cover_all_14_dmma_instances():
    seen = set()
    for inst in R.DMMA_INSTANCES:
        seen |= _instances(R.dmma_instance(*inst))
    assert len(R.DMMA_INSTANCES) == 14
    assert seen == set(R.DMMA_INSTANCES)


def test_mixed_set_layout():
    """Two blocks of >= 6 consumer warps (producers at warps 3 and 7), a padding item, items
    starting at nz tile 4, every wavevector once."""
    n = R.dmma_mixed()
    plan = _lib.sq_plan(n)
    items = _lib.sq_plan_items(n)["mma"]
    W = plan["warps_per_block"]
    assert W >= 6 and len(items) % W == 0 and len(items) // W >= 2
    assert items[:, 3].sum() >= 1                            # padding
    assert (items[items[:, 3] == 1][:, :2] == 0).all()
    assert (items[:, 2] == 4).any()                          # t0 = 4
    assert len(_instances(n)) >= 5
    assert (plan["coverage"] == 1).all() and plan["pair_rule_violations"] == 0


@pytest.mark.parametrize("second", [False, True])
def test_scalar_builders_run_each_R(second):
    for r in range(1, 9):
        warps = _lib.sq_plan_items(R.scalar_instance(r, second))["lattice_r"].tolist()
        assert warps == ([8, r] if second else [r])


def _scalar_smem(nm, elem=8):
    # launch_lattice: two buffers of kPS = 32 particles x lattice_row_elems(nmax) elements
    oy = 2 * (nm[0] + 1)
    oz = (oy + 2 * (nm[1] + 1) + 3) // 4 * 4
    return 2 * elem * 32 * (oz + 2 * ((nm[2] + 8) // 8 * 8))


def test_limit_sets_sit_on_both_sides_of_the_table_limits():
    dmma = lambda *s: _lib.sq_plan(R.limit_set(*s))["smem_bytes"]       # noqa: E731
    assert dmma(47, 47, 47) <= 200 * 1024 < dmma(48, 48, 48)
    assert _scalar_smem((72, 72, 72)) <= 227 * 1024 < _scalar_smem((73, 73, 73))
    assert _lib.sq_plan(R.deep_set(150, 7))["smem_bytes"] <= 200 * 1024
    assert _lib.sq_plan(R.deep_set(200, 0))["smem_bytes"] > 200 * 1024
    assert _scalar_smem((200, 0, 0)) <= 227 * 1024
    for s in [(47, 47, 47), (48, 48, 48), (72, 72, 72), (73, 73, 73)]:
        assert R.limit_set(*s).max(axis=0).tolist() == list(s)
    assert R.deep_set(150, 7).max(axis=0).tolist() == [150, 0, 7]
    assert R.deep_set(200, 0).max(axis=0).tolist() == [200, 0, 0]


_CASES = [("inst44", R.dmma_instance(4, 4)), ("mixed", R.dmma_mixed()),
          ("scalar8", R.scalar_instance(8, True)), ("lim47", R.limit_set(47, 47, 47)),
          ("lim72", R.limit_set(72, 72, 72)), ("lim73", R.limit_set(73, 73, 73)),
          ("deep150", R.deep_set(150, 7)), ("deep200", R.deep_set(200, 0))]


@pytest.mark.parametrize("kernel", ["lattice_dmma", "lattice_fp64", "general_fp64"])
def test_fp64_bounds_are_not_vacuous(kernel):
    """The GPU test's fp64 cases: S(q) bound <= 1e-10 per frame (S normalised by N), i.e.
    well under the 1e-9 relative the rest of the suite asks, and the reference's own error
    more than 1000x below every rho bound."""
    pos, b = R.particles()
    for name, n in _CASES:
        S, dS, _, _, margin = R.expected_s(pos, n, b, kernel)
        assert margin > 1000, (name, margin)
        assert dS.max() / (R.N_TOTAL * len(pos)) <= 1e-10, name


def test_float64_entry_bound_is_set_by_the_coordinate_split():
    """Far from the origin (|r| ~ 10^3, 90 box lengths) the float64 entry point's coordinate
    error 2^-48 |r| dominates; its S bound is still > 100x below what a float32 copy of the
    coordinates costs (phase error up to 2^-24 |q||r| per term)."""
    pos, b = R.particles(seed=7, offset=1000.0, dtype=np.float64)
    n = R.deep_set(150, 7)
    for kernel in ("lattice_dmma", "lattice_fp64"):
        S, dS, _, _, margin = R.expected_s(pos, n, b, kernel, R.COORD_REL_F64)
        assert margin > 1000
        S32, dS32, _, _, _ = R.expected_s(pos, n, b, kernel, R.UF)
        assert dS.max() * 100 < dS32.max()
        assert dS.max() / (R.N_TOTAL * len(pos)) < 1e-7


def test_rho_ref_against_a_float64_sum():
    """rho_ref agrees with a plain float64 sum within that sum's own error (phase
    arguments |q.r| u each, sincos and the sum of N terms)."""
    pos, b = R.particles(frames=1)
    x = pos[0].astype(np.float64)
    for n in (R.dmma_instance(4, 4), R.deep_set(200, 0)):
        ref = R.rho_ref(x, n, b).astype(np.complex128)
        arg = x @ (n * b).T
        plain = np.exp(1j * arg).sum(axis=0)
        err64 = (np.abs(arg).sum(axis=0) * 3 * R.U + len(x) * 6 * R.U
                 + np.sqrt(2) * R.U * len(x) ** 2)
        assert (np.abs(plain - ref) <= err64).all()
        # and it is not the same arithmetic: the two differ where the phases are large
        assert np.abs(plain - ref).max() > 0


def test_rho_bound_grows_with_recurrence_depth_and_coordinates():
    pos, b = R.particles(frames=1)
    n = np.array([(0, 0, 1), (0, 0, 40), (0, 0, 160)], dtype=np.int32)
    for kernel in ("lattice_dmma", "lattice_fp64", "lattice_fp32", "general_fp64"):
        d = R.rho_bound(kernel, pos[0], n, b)
        assert d[0] < d[1] < d[2]
        assert (R.rho_bound(kernel, pos[0] + 100, n, b) > d).all()
