#!/usr/bin/env python
"""fp32 filter of the triclinic cell list against its fp64 kernel, on device-resident
frames: one JSON line with

- the device name and power limit (read in this call);
- per workload, arith "off" (rdf_tri_cells_kernel) and "auto" (rdf_tri_cells_filter_kernel)
  timed alternately, three rounds each: us per frame of the whole pipeline (pack, wrap,
  sort, pair kernel; CUDA events of mdh_kernel_time) over 128 frames after a warm-up,
  candidates per second, the fraction of candidates re-evaluated exactly, and whether the
  counts of the two are equal;
- workloads: the 500,000-particle rhombic dodecahedron and truncated octahedron of
  tools/tri_cells_speed.py (rho* = 0.8, range (0, 2.5), 100 bins), the 300,000-particle
  hexagonal slab of tools/slab_cells_speed.py (drop_axis = 2), and the orthorhombic cell
  list on cfg3 as the yardstick (its own filter, arith "off" vs "auto").

Usage: tri_cells_filter_speed.py [OUT.json].  Needs a CUDA device; there is no fallback."""
import json
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import torch  # noqa: E402

import slab_cells_speed as slab  # noqa: E402
import tri_cells_speed as tri  # noqa: E402
from mdhelper_b200 import _lib, synthetic  # noqa: E402
from mdhelper_b200.analysis._binning import squared_thresholds  # noqa: E402
from mdhelper_b200.analysis._triclinic import triclinic_vectors  # noqa: E402

ROUNDS = 3


def time_tri(dev, cells, n, arith, per_call=8, calls=16, warm=2, drop=None):
    ctx = _lib.Context(0)
    ctx.rdf_set_filter(arith)
    ctx.rdf_configure(n, n, True, squared_thresholds(tri.BINS, tri.RANGE), *tri.RANGE,
                      mode="cells", drop_axis=drop)
    frames = len(cells)

    def call(k):
        f0 = (k * per_call) % (frames - per_call + 1)
        p = dev.data_ptr() + 12 * n * f0
        ctx.rdf_accumulate_triclinic(p, 3 * n, p, 3 * n, cells[f0:f0 + per_call], per_call,
                                     device=True)
    for k in range(warm):
        call(k)
    ctx.sync()
    ctx.rdf_reset()
    ctx.kernel_time(reset=True)
    for k in range(calls):
        call(k)
    ctx.sync()
    ms, _, _, _ = ctx.kernel_time(reset=True)
    counts = ctx.rdf_fetch()
    ev = ctx.rdf_pair_evaluations()
    st = ctx.rdf_filter_stats()
    ctx.close()
    nf = per_call * calls
    return {"us_per_frame": 1e3 * ms / nf, "candidates_per_s": ev / (ms * 1e-3),
            "candidates_per_frame": ev / nf,
            "exact_fraction": st["triclinic_exact_pairs"] / max(ev, 1),
            "triclinic_frames": st["triclinic_frames"],
            "declined_frames": st["declined_frames"]}, counts


def compare(fn):
    """Alternate off / auto ROUNDS times; the median of each, counts compared per round."""
    runs = {"off": [], "auto": []}
    equal = True
    for _ in range(ROUNDS):
        off, c_off = fn("off")
        auto, c_auto = fn("auto")
        runs["off"].append(off)
        runs["auto"].append(auto)
        equal = equal and bool(np.array_equal(c_off, c_auto)) and bool(c_off.sum() > 0)
    med = {k: sorted(v, key=lambda r: r["us_per_frame"])[ROUNDS // 2] for k, v in runs.items()}
    return {"off": med["off"], "auto": med["auto"],
            "us_per_frame_rounds": {k: [r["us_per_frame"] for r in v] for k, v in runs.items()},
            "speedup": med["off"]["us_per_frame"] / med["auto"]["us_per_frame"],
            "counts_equal": equal}


_CFG3 = {}


def ortho_cfg3(arith):
    if not _CFG3:
        u = synthetic.lj_fluid(500_000, 32, seed=20260003, pinned=False)
        _CFG3["dev"] = torch.from_numpy(u.trajectory.coordinates).cuda()
        _CFG3["boxes"] = np.ascontiguousarray(u.trajectory.unitcells[:, :3])
    dev, boxes = _CFG3["dev"], _CFG3["boxes"]
    F, n = dev.shape[:2]
    ctx = _lib.Context(0)
    ctx.rdf_set_filter(arith)
    ctx.rdf_configure(n, n, True, squared_thresholds(tri.BINS, tri.RANGE), *tri.RANGE,
                      mode="cells")

    def call(k):
        f0 = (k * 16) % (F - 16 + 1)
        ctx.rdf_accumulate(dev.data_ptr() + 12 * n * f0, 3 * n, None, 0, boxes[f0:f0 + 16], 16,
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
    counts = ctx.rdf_fetch()
    ctx.close()
    return {"us_per_frame": 1e3 * ms / 128, "candidates_per_s": ev / (ms * 1e-3)}, counts


def main():
    if not torch.cuda.is_available():
        raise SystemExit("tri_cells_filter_speed.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = tri.device_info()
    out = {"device": name, "power_limit": power, "range": list(tri.RANGE), "n_bins": tri.BINS}
    for key, angles, seed in (("rhombic_dodecahedron", (60.0, 60.0, 90.0), 1),
                              ("truncated_octahedron", (70.53, 109.47, 70.53), 2)):
        dims, cells, pos = tri.tri_system(angles, seed)
        dev = torch.from_numpy(pos).cuda()
        out[key] = compare(lambda a: time_tri(dev, cells, tri.N, a))
        out[key].update({"n": tri.N, "dims": [float(v) for v in dims]})
        del dev
    dims, pos = slab.slab(120.0, 2)
    box = dims[:3].copy()
    box[2] = box.max()                         # the reference's widened edge (drop_axis = 2)
    cell = triclinic_vectors(np.array([*box, *dims[3:]], np.float32))
    dev = torch.from_numpy(pos).cuda()
    cells = np.stack([cell] * len(pos)).astype(np.float32)
    out["hexagonal_slab"] = compare(lambda a: time_tri(dev, cells, slab.N, a, drop=2))
    out["hexagonal_slab"].update({"n": slab.N, "dims": [float(v) for v in dims],
                                  "drop_axis": 2})
    del dev
    out["ortho_cells_cfg3"] = compare(ortho_cfg3)
    print(json.dumps(out), flush=True)
    if len(sys.argv) > 1:                      # optional: also write the line to a file
        pathlib.Path(sys.argv[1]).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
