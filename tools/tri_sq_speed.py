#!/usr/bin/env python
"""S(q) on the reciprocal lattice of a triclinic cell against the orthorhombic cfg4 rate, on
device-resident frames: one JSON line with

- the device name and power limit (read in this call);
- per case: N_q, the kernel the library chose, frames/s and terms/s (N * N_q per frame) from
  the CUDA events of mdh_kernel_time (every kernel of an accumulate call, the fractional-
  coordinate map and the float32 + remainder split included) and from the host clock
  around synchronised calls, after a warm-up;
- cases, all with N = 50,000 particles at rho* = 0.8 and 256 frames on the device:
    edges_cfg4        cfg4 of bench.py: cubic box, reciprocal="edges", n_max = 16
                      (q_max = 2 pi 16 / L, N_q = 2,446);
    cell_rd           the same number density in a rhombic dodecahedron (60, 60, 90),
                      reciprocal="cell", q_max chosen so that N_q is closest to 2,446;
    edges_general_rd  the Cartesian wavevectors of cell_rd passed as wavevectors= with
                      reciprocal="edges": off the edge-length lattice, so the general kernel.

Usage: tri_sq_speed.py [OUT.json].  Needs a CUDA device; there is no fallback."""
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from mdhelper_b200 import _lib, synthetic  # noqa: E402
from mdhelper_b200.analysis._triclinic import box_volume, triclinic_vectors  # noqa: E402
from mdhelper_b200.analysis.structure import StructureFactor  # noqa: E402
from mdhelper_b200.universe import SyntheticUniverse  # noqa: E402

N, FRAMES, RHO, NQ_CFG4 = 50_000, 256, 0.8, 2446
RD = (60.0, 60.0, 90.0)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = (s.strip() for s in q.split(","))
    return name, power


def rd_universe():
    """N particles uniform in a rhombic dodecahedron of volume N / rho."""
    unit = box_volume(np.array([1.0, 1.0, 1.0, *RD]))
    a = (N / RHO / unit) ** (1 / 3)
    dims = np.array([a, a, a, *RD], np.float32)
    h = triclinic_vectors(dims).astype(np.float64)
    rng = np.random.default_rng(20261022)
    pos = (rng.random((FRAMES, N, 3)) @ h).astype(np.float32)
    return SyntheticUniverse(pos, dims)


def rd_q_max(u):
    """q_max of the cell grid whose N_q is closest to cfg4's (ties: the smaller)."""
    q = np.sort(StructureFactor(u.atoms, n_points=32, reciprocal="cell",
                                verbose=False)._wavenumbers)
    cut = np.unique(q)
    n_q = np.searchsorted(q, cut, side="right")
    return float(cut[int(np.argmin(np.abs(n_q - NQ_CFG4)))])


def time_case(sf, dev, per_call=16, min_s=2.0):
    ctx = _lib.Context(0)
    kernel = None if sf._lattice_n is not None else "general_fp64"
    ctx.sq_configure(N, [0, N], sf._kvectors, [(-1, -1)], lattice_n=sf._lattice_n,
                     lattice_b=sf._lattice_b, mode=kernel or "auto")
    if sf._cell is not None:
        ctx.sq_set_cell(sf._cell)
    base = dev.data_ptr()

    def call(k):
        f0 = (k * per_call) % FRAMES
        ctx.sq_accumulate(base + 12 * N * f0, 3 * N, per_call, device=True)

    call(0)                                    # warm-up: modules, work items, buffers
    ctx.sync()
    ctx.kernel_time(reset=True)
    calls, t0 = 0, time.perf_counter()
    while calls < 3 or time.perf_counter() - t0 < min_s:
        call(calls)
        calls += 1
        if calls % 4 == 0:
            ctx.sync()
    ctx.sync()
    wall = time.perf_counter() - t0
    _, _, ms, _ = ctx.kernel_time(reset=True)
    frames = calls * per_call
    n_q = len(sf._kvectors)
    out = {"n_q": n_q, "kernel": ctx.sq_kernel(), "frames": frames,
           "frames_per_s": frames / (ms * 1e-3), "terms_per_s": frames * N * n_q / (ms * 1e-3),
           "frames_per_s_wall": frames / wall}
    ctx.close()
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit("tri_sq_speed.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = device_info()
    out = {"device": name, "power_limit": power, "n": N, "rho": RHO}

    u = synthetic.lj_fluid(N, FRAMES, seed=20260004, pinned=False)
    L = float(u.trajectory.unitcells[0, 0])
    dev = torch.from_numpy(u.trajectory.coordinates).cuda()
    sf = StructureFactor(u.atoms, n_points=32, q_max=2 * np.pi * 16 / L, verbose=False)
    out["edges_cfg4"] = time_case(sf, dev)
    out["edges_cfg4"]["dims"] = [float(v) for v in u.dimensions]
    del dev

    u = rd_universe()
    q_max = rd_q_max(u)
    dev = torch.from_numpy(u.trajectory.coordinates).cuda()
    sf = StructureFactor(u.atoms, n_points=32, q_max=q_max, reciprocal="cell", verbose=False)
    out["cell_rd"] = time_case(sf, dev)
    out["cell_rd"].update({"dims": [float(v) for v in u.dimensions], "q_max": q_max})
    ge = StructureFactor(u.atoms, wavevectors=sf._wavevectors, verbose=False)
    out["edges_general_rd"] = time_case(ge, dev, per_call=4)
    del dev
    e, c, g = out["edges_cfg4"], out["cell_rd"], out["edges_general_rd"]
    out["cell_over_edges_terms_per_s"] = c["terms_per_s"] / e["terms_per_s"]
    out["cell_over_general_terms_per_s"] = c["terms_per_s"] / g["terms_per_s"]
    print(json.dumps(out), flush=True)
    if len(sys.argv) > 1:                      # optional: also write the line to a file
        pathlib.Path(sys.argv[1]).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
