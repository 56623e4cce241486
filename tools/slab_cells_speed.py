#!/usr/bin/env python
"""Two-dimensional RDF (drop_axis=2) of one particle layer on device-resident frames: one
JSON line with

- the device name and power limit (read in this call);
- an orthorhombic and a hexagonal (90, 90, 120 degrees) slab of 300,000 particles in one
  layer, areal density 0.8 (a jittered lattice: no overlaps), range (0, 2.5), 100 bins;
- per slab: us per frame of the whole cell-list pipeline (CUDA events of mdh_kernel_time;
  the orthorhombic slab with the fp32 filter and with fp64 for every pair), 128 timed
  frames after a warm-up, and its candidate evaluations per second; the all-pairs kernel
  on one frame, with its counts compared to the cell list's on that frame;
- the three-dimensional orthorhombic cell list on a 300,000-particle fluid (rho* = 0.8,
  same range and bins) in the same call, as a yardstick for the per-candidate rate.

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

from mdhelper_b200 import _lib  # noqa: E402
from mdhelper_b200.analysis._binning import squared_thresholds  # noqa: E402
from mdhelper_b200.analysis._triclinic import triclinic_vectors  # noqa: E402

N, RHO2, RHO3, RANGE, BINS = 300_000, 0.8, 0.8, (0.0, 2.5), 100
FRAMES, PER_CALL, CALLS = 8, 8, 16          # 128 timed frames
LZ = 40.0                                    # slab thickness (the dropped edge)


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60)
        power = out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def jittered(frac_grid_dims, n, seed):
    """n points of a jittered lattice in fractional coordinates, FRAMES frames."""
    d = len(frac_grid_dims)
    m = int(np.ceil(n ** (1 / d)))
    g = np.stack(np.meshgrid(*[np.arange(m)] * d, indexing="ij"), -1).reshape(-1, d)[:n]
    rng = np.random.default_rng(seed)
    return [(g + 0.5 + rng.uniform(-0.2, 0.2, g.shape)) / m for _ in range(FRAMES)]


def slab(gamma, seed):
    """N particles in one layer of a cell (L, L, LZ, 90, 90, gamma); z spread over 1."""
    unit = triclinic_vectors(np.array([1, 1, 1, 90, 90, gamma], np.float32)).astype(np.float64)
    area1 = unit[0, 0] * unit[1, 1]
    L = np.sqrt(N / RHO2 / area1)
    dims = np.array([L, L, LZ, 90, 90, gamma], np.float32)
    h = triclinic_vectors(dims).astype(np.float64)
    rng = np.random.default_rng(seed + 100)
    pos = np.empty((FRAMES, N, 3), np.float32)
    for f, fr in enumerate(jittered((1, 1), N, seed)):
        xy = fr @ h[:2, :2]
        pos[f] = np.column_stack([xy, 0.5 * LZ + rng.uniform(-0.5, 0.5, N)]).astype(np.float32)
    return dims, pos


def bulk(seed):
    L = (N / RHO3) ** (1 / 3)
    pos = np.stack([(fr * L).astype(np.float32) for fr in jittered((1, 1, 1), N, seed)])
    return np.array([L, L, L, 90, 90, 90], np.float32), pos


def run(dev, dims, mode, drop, frames_per_call, calls, warm=2, arith="auto"):
    """Timed accumulate calls of `frames_per_call` device-resident frames each."""
    ortho = bool(np.all(dims[3:] == 90))
    box = dims[:3].copy()
    if drop is not None:
        box[drop] = box.max()                  # the reference's widened edge
    cell = triclinic_vectors(np.array([*box, *dims[3:]], np.float32))
    ctx = _lib.Context(0)
    ctx.rdf_set_filter(arith)
    ctx.rdf_configure(N, N, True, squared_thresholds(BINS, RANGE), *RANGE, mode=mode,
                      drop_axis=drop)

    def call(k):
        f0 = (k * frames_per_call) % (FRAMES - frames_per_call + 1)
        p = dev.data_ptr() + 12 * N * f0
        if ortho:
            ctx.rdf_accumulate(p, 3 * N, None, 0, np.stack([box] * frames_per_call),
                               frames_per_call, device=True)
        else:
            ctx.rdf_accumulate_triclinic(p, 3 * N, p, 3 * N, np.stack([cell] * frames_per_call),
                                         frames_per_call, device=True)
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


def main():
    if not torch.cuda.is_available():
        raise SystemExit("slab_cells_speed.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = device_info()
    out = {"device": name, "power_limit": power, "n": N, "areal_density": RHO2,
           "range": list(RANGE), "n_bins": BINS, "drop_axis": 2}
    for key, gamma, seed in (("orthorhombic_slab", 90.0, 1), ("hexagonal_slab", 120.0, 2)):
        dims, pos = slab(gamma, seed)
        dev = torch.from_numpy(pos).cuda()
        box = dims[:3].copy()
        box[2] = box.max()
        grid, margin = _lib.cells_grid(
            triclinic_vectors(np.array([*box, *dims[3:]], np.float32)), RANGE[1], N, 2)
        res, _ = run(dev, dims, "cells", 2, PER_CALL, CALLS)
        one_cells, c1 = run(dev, dims, "cells", 2, 1, 1, warm=1)
        one_all, c2 = run(dev, dims, "allpairs", 2, 1, 1, warm=0)
        res.update({"dims": [float(v) for v in dims], "grid": list(grid), "margin": margin,
                    "allpairs_us_one_frame": one_all["us_per_frame"],
                    "allpairs_evaluations_per_s": one_all["evaluations_per_s"],
                    "cells_us_one_frame": one_cells["us_per_frame"],
                    "counts_equal": bool(np.array_equal(c1, c2)),
                    "pairs_binned_one_frame": int(c1.sum()),
                    "speedup_vs_allpairs": one_all["us_per_frame"] / res["us_per_frame"]})
        if gamma == 90.0:
            res["fp64"], c3 = run(dev, dims, "cells", 2, PER_CALL, CALLS, arith="off")
        out[key] = res
        del dev
    dims, pos = bulk(3)
    dev = torch.from_numpy(pos).cuda()
    out["bulk_3d_cells"], _ = run(dev, dims, "cells", None, PER_CALL, CALLS)
    out["bulk_3d_cells"]["fp64"], _ = run(dev, dims, "cells", None, PER_CALL, CALLS,
                                          arith="off")
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
