#!/usr/bin/env python
"""fp32 filter of the triclinic all-pairs path on device-resident frames: one JSON line
on stdout with

- the device name and power limit (read in this call);
- cfg2's 20,000 ions at rho* = 0.8 in a rhombic dodecahedron (d ~ 32.8, R ~ 11.6), two
  groups of 10,000, 201 bins, range (0, 11): ms per frame and ordered pairs per second with
  arith "off" (27 images in fp64 for every pair) and "auto" (the filter), alternated in this
  call (CUDA events around each accumulate call, 8 frames per call, after a warm-up), with
  the counts of both compared;
- the orthorhombic cfg2 all-pairs filter (cube of the same volume, arith "auto") in the
  same call, as the yardstick;
- an N sweep at range (0, 2.5), one group, rho* = 0.8, rhombic dodecahedron: ms per frame
  of the filtered all-pairs kernel and of the triclinic cell list, and where they cross.

Needs a CUDA device; there is no fallback."""
import json
import pathlib
import subprocess
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from mdhelper_b200 import _lib  # noqa: E402
from mdhelper_b200.analysis._binning import squared_thresholds  # noqa: E402
from mdhelper_b200.analysis._triclinic import triclinic_vectors  # noqa: E402

RD = (60.0, 60.0, 90.0)
FRAMES = 8


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=60)
        power = out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def rd_cell(n, rho=0.8):
    unit = triclinic_vectors(np.array([1, 1, 1, *RD], np.float32)).astype(np.float64)
    L = (n / rho / abs(np.linalg.det(unit))) ** (1 / 3)
    return triclinic_vectors(np.array([L, L, L, *RD], np.float32)).astype(np.float32)


def positions(n, h, seed):
    rng = np.random.default_rng(seed)
    p = (rng.random((FRAMES, n, 3)) @ h.astype(np.float64)).astype(np.float32)
    return torch.from_numpy(p).cuda()


def timed(fn, reps):
    fn()                                    # warm-up (module load, buffers)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), ts


def tri_run(p1, p2, cells, n_bins, rng_, arith, mode="allpairs"):
    ctx = _lib.Context(0)
    n1, n2 = p1.shape[1], (p1 if p2 is None else p2).shape[1]
    ctx.rdf_set_filter(arith)
    ctx.rdf_configure(n1, n2, p2 is None, squared_thresholds(n_bins, rng_), rng_[0], rng_[1],
                      mode=mode)
    b = p1 if p2 is None else p2

    def go():
        ctx.rdf_reset()
        ctx.rdf_accumulate_triclinic(p1, 3 * n1, b, 3 * n2, cells, FRAMES, device=True)
    return ctx, go


def main():
    assert torch.cuda.is_available(), "needs a CUDA device"
    name, power = device_info()
    out = {"device": name, "power_limit": power, "frames_per_call": FRAMES}

    # cfg2 in a rhombic dodecahedron, off vs auto alternated
    h = rd_cell(20_000)
    cells = np.stack([h] * FRAMES)
    p1, p2 = positions(10_000, h, 1), positions(10_000, h, 2)
    runs = {a: tri_run(p1, p2, cells, 201, (0.0, 11.0), a) for a in ("off", "auto")}
    med = {"off": [], "auto": []}
    for _ in range(3):
        for a, (ctx, go) in runs.items():
            m, _ = timed(go, 3 if a == "off" else 10)
            med[a].append(m)
    counts = {a: ctx.rdf_fetch() for a, (ctx, _) in runs.items()}
    stats = runs["auto"][0].rdf_filter_stats()
    pairs = 10_000 * 10_000 * FRAMES
    cfg2 = {"cell_diag": [float(h[0, 0]), float(h[1, 1]), float(h[2, 2])],
            "R": 0.5 * float(min(h[0, 0], h[1, 1], h[2, 2])),
            "counts_equal": bool(np.array_equal(counts["off"], counts["auto"])),
            "filter_stats": stats}
    for a in ("off", "auto"):
        ms = float(np.median(med[a]))
        cfg2[a] = {"ms_per_frame": ms / FRAMES, "ordered_pairs_per_s": pairs / (ms * 1e-3),
                   "call_medians_ms": med[a]}
    cfg2["speedup"] = cfg2["off"]["ms_per_frame"] / cfg2["auto"]["ms_per_frame"]
    for ctx, _ in runs.values():
        ctx.close()
    out["cfg2_rd"] = cfg2

    # yardstick: the orthorhombic filter on cfg2 (cube of the same volume)
    L = float(abs(np.linalg.det(h.astype(np.float64))) ** (1 / 3))
    rng = np.random.default_rng(3)
    q1 = torch.from_numpy((rng.random((FRAMES, 10_000, 3)) * L).astype(np.float32)).cuda()
    q2 = torch.from_numpy((rng.random((FRAMES, 10_000, 3)) * L).astype(np.float32)).cuda()
    box = np.full((FRAMES, 3), L, np.float32)
    ctx = _lib.Context(0)
    ctx.rdf_configure(10_000, 10_000, False, squared_thresholds(201, (0.0, 11.0)), 0.0, 11.0,
                      mode="allpairs")

    def go_o():
        ctx.rdf_reset()
        ctx.rdf_accumulate(q1, 30_000, q2, 30_000, box, FRAMES, device=True)
    m, _ = timed(go_o, 10)
    ctx.close()
    out["cfg2_ortho"] = {"ms_per_frame": m / FRAMES, "pairs_per_s": pairs / (m * 1e-3)}

    # N sweep at (0, 2.5): filtered all pairs against the triclinic cell list
    sweep = []
    for n in (2_000, 5_000, 10_000, 20_000, 50_000, 100_000):
        h = rd_cell(n)
        cells = np.stack([h] * FRAMES)
        p = positions(n, h, 4)
        row = {"n": n}
        got = {}
        for mode in ("allpairs", "cells"):
            ctx, go = tri_run(p, None, cells, 100, (0.0, 2.5), "auto", mode=mode)
            m, _ = timed(go, 5)
            got[mode] = ctx.rdf_fetch()
            row[mode + "_ms_per_frame"] = m / FRAMES
            ctx.close()
        row["counts_equal"] = bool(np.array_equal(got["allpairs"], got["cells"]))
        sweep.append(row)
    out["sweep_0_2p5"] = sweep
    cross = [r["n"] for r in sweep if r["cells_ms_per_frame"] < r["allpairs_ms_per_frame"]]
    out["cells_faster_from_n"] = min(cross) if cross else None

    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
