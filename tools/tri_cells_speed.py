#!/usr/bin/env python
"""Triclinic cell-list pipeline on device-resident frames: one JSON line with

- the device name and power limit (read in this call);
- us per frame of the whole triclinic cell-list pipeline (pack, wrap, sort, pair kernel;
  CUDA events of mdh_kernel_time) for a 500,000-particle LJ-like fluid at rho* = 0.8,
  range (0, 2.5), 100 bins, in a rhombic dodecahedron (60, 60, 90 degrees) and a truncated
  octahedron (70.53, 109.47, 70.53), >= 100 frames after a warm-up, and its candidate
  evaluations per second;
- the all-pairs triclinic kernel on one frame of the same system, with its counts
  compared to the cell list's on that frame;
- the orthorhombic fp64 cell list (mode="cells", arith="off") on cfg3, measured in the
  same call, as a yardstick for the per-candidate rate.

Needs a CUDA device; there is no fallback."""
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
from mdhelper_b200.analysis._binning import squared_thresholds  # noqa: E402
from mdhelper_b200.analysis._triclinic import triclinic_vectors  # noqa: E402

N, RHO, RANGE, BINS = 500_000, 0.8, (0.0, 2.5), 100
FRAMES, PER_CALL = 8, 8            # device-resident frames, frames per accumulate call
CALLS = 16                         # 128 timed frames


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60)
        power = out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def tri_system(angles, seed):
    """N particles, rho* = 0.8, equal edge lengths with the given angles; the positions
    are a jittered lattice in fractional coordinates (LJ-like: no overlaps), FRAMES
    frames."""
    unit = triclinic_vectors(np.array([1, 1, 1, *angles], np.float32)).astype(np.float64)
    L = (N / RHO / abs(np.linalg.det(unit))) ** (1 / 3)
    dims = np.array([L, L, L, *angles], np.float32)
    h = triclinic_vectors(dims).astype(np.float64)
    m = int(np.ceil(N ** (1 / 3)))
    g = np.stack(np.meshgrid(*[np.arange(m)] * 3, indexing="ij"), -1).reshape(-1, 3)[:N]
    rng = np.random.default_rng(seed)
    pos = np.empty((FRAMES, N, 3), np.float32)
    for f in range(FRAMES):
        frac = (g + 0.5 + rng.uniform(-0.2, 0.2, g.shape)) / m
        pos[f] = (frac @ h).astype(np.float32)
    return dims, np.stack([h] * FRAMES).astype(np.float32), pos


def time_tri(dev, cells, mode, frames_per_call, calls, warm=2):
    ctx = _lib.Context(0)
    ctx.rdf_configure(N, N, True, squared_thresholds(BINS, RANGE), *RANGE, mode=mode)

    def call(k):
        f0 = (k * frames_per_call) % (FRAMES - frames_per_call + 1)
        ctx.rdf_accumulate_triclinic(dev.data_ptr() + 12 * N * f0, 3 * N,
                                     dev.data_ptr() + 12 * N * f0, 3 * N,
                                     cells[f0:f0 + frames_per_call], frames_per_call,
                                     device=True)
    for k in range(warm):
        call(k)
    ctx.sync()
    ctx.rdf_reset()
    ctx.kernel_time(reset=True)
    t0 = time.perf_counter()
    for k in range(calls):
        call(k)
    ctx.sync()
    wall = time.perf_counter() - t0
    ms, _, _, _ = ctx.kernel_time(reset=True)
    counts = ctx.rdf_fetch()
    ev = ctx.rdf_pair_evaluations()
    ctx.close()
    frames = frames_per_call * calls
    return {"frames": frames, "us_per_frame": 1e3 * ms / frames,
            "wall_us_per_frame": 1e6 * wall / frames, "evaluations_per_frame": ev / frames,
            "evaluations_per_s": ev / (ms * 1e-3)}, counts


def ortho_cfg3():
    u = synthetic.lj_fluid(500_000, 32, seed=20260003, pinned=False)
    coords = u.trajectory.coordinates
    F = coords.shape[0]
    dev = torch.from_numpy(coords).cuda()
    boxes = np.ascontiguousarray(u.trajectory.unitcells[:, :3])
    ctx = _lib.Context(0)
    ctx.rdf_set_filter("off")
    ctx.rdf_configure(N, N, True, squared_thresholds(BINS, RANGE), *RANGE, mode="cells")

    def call(k):
        f0 = (k * 16) % (F - 16 + 1)
        ctx.rdf_accumulate(dev.data_ptr() + 12 * N * f0, 3 * N, None, 0, boxes[f0:f0 + 16], 16,
                           device=True)
    for k in range(2):
        call(k)
    ctx.sync()
    ctx.rdf_reset()
    ctx.kernel_time(reset=True)
    for k in range(8):
        call(k)
    ctx.sync()
    ms, _, _, _ = ctx.kernel_time(reset=True)
    ev = ctx.rdf_pair_evaluations()
    ctx.close()
    return {"frames": 128, "us_per_frame": 1e3 * ms / 128, "evaluations_per_frame": ev / 128,
            "evaluations_per_s": ev / (ms * 1e-3)}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("tri_cells_speed.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = device_info()
    out = {"device": name, "power_limit": power, "n": N, "rho": RHO, "range": list(RANGE),
           "n_bins": BINS}
    for key, angles, seed in (("rhombic_dodecahedron", (60.0, 60.0, 90.0), 1),
                              ("truncated_octahedron", (70.53, 109.47, 70.53), 2)):
        dims, cells, pos = tri_system(angles, seed)
        dev = torch.from_numpy(pos).cuda()
        grid, margin = _lib.triclinic_grid(cells[0], RANGE[1], N)
        res, _ = time_tri(dev, cells, "cells", PER_CALL, CALLS)
        one_cells, c1 = time_tri(dev, cells, "cells", 1, 1, warm=1)
        one_all, c2 = time_tri(dev, cells, "allpairs", 1, 1, warm=0)
        res.update({"dims": [float(v) for v in dims], "grid": list(grid), "margin": margin,
                    "allpairs_us_one_frame": one_all["us_per_frame"],
                    "cells_us_one_frame": one_cells["us_per_frame"],
                    "counts_equal": bool(np.array_equal(c1, c2)),
                    "pairs_binned_one_frame": int(c1.sum()),
                    "speedup_vs_allpairs": one_all["us_per_frame"] / res["us_per_frame"]})
        out[key] = res
        del dev
    out["ortho_fp64_cells_cfg3"] = ortho_cfg3()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
