#!/usr/bin/env python
"""
bench.py -- hot-path benchmark (contract: one JSON line on stdout from rank 0).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps K --warmup W      # CPU reference arm

Headline workload (BASELINE.json configs[1], SURVEY.md section 8(d) "cfg2"): two-group
cation-anion partial RDF of a 20,000-ion electrolyte, n_bins=201, range (0, 14.5), 2,000
synthetic frames.  One "step" = one pass of the pair-histogram hot path over the whole
2,000-frame trajectory (ten C-ABI calls of 200 frames); under torchrun every rank brings
its own trajectory (weak scaling).

* ``value``      pairs binned / s, coordinates already resident in HBM, device time (CUDA
                 events on the launching stream), max over ranks.
* ``e2e``        the same metric through the public class
                 ``RadialDistributionFunction(cations, anions).run()`` from pinned HOST
                 memory (H2D of every frame and D2H of the counts inside the timed region).
* ``roofline``   the kernel that runs by default is the fp32-filter pair kernel
                 (rdf_filter.cu: counts identical to the reference's fp64 arithmetic,
                 uncertain pairs re-evaluated in fp64): pair evaluations/s x 16 FP32
                 operations per evaluation over the measured packed-FP32 rate x SM count x
                 the SM clock sampled during the run; beside it
                 ``fp64_pipe_equivalent_frac``, the same rate against the bound of a kernel
                 that executes the reference's 21 FP64 instructions per pair.  ``--arith
                 off`` benches that kernel (FP64-pipe roofline).
* ``cpu_baseline`` the restated reference CPU path (oracle/: C distances + real
                 numpy.histogram), serial and frame-parallel over all host cores, on a
                 bounded sample of the same frames.
* ``secondary``  the S(q) half of BASELINE's metric: frames/s of the direct-sum structure
                 factor for N=50,000, N_q=2,446 (configs[3]; step = its 1,000 frames) with
                 its own roofline, e2e and CPU baseline.  ``--impl reference`` carries the
                 CPU S(q) rate in the same place.
* ``strong``     the named configurations at their named scale, STRONG scaling: a fixed
                 frame list -- cfg4: 1,000 frames of S(q); cfg3: 1,000 frames of the cut-off
                 RDF of 500,000 particles; cfg5: 500 frames of the combined RDF + S(q) pass
                 over 1,000,000 beads -- through ``run()`` / ``CombinedAnalysis.run()``,
                 split over the ranks as the reference splits its frame list
                 (base.py:433-441), host memory -> results.  Under torchrun rank 0 then
                 recomputes the whole span alone and compares (``multi_gpu_parity``:
                 integer counts identical, S(q) within 1e-12 relative).

Multi-GPU: frames shard over ranks, no data-path collective; one NCCL all-reduce of the
accumulators at the end, inside the timed region.

``--dump-outputs DIR`` writes, after the timed steps, what the last timed step of each
measured path returned to its caller as ``DIR/<name>.npy`` (float64, a few kB in all):
``rdf_counts`` (headline), ``rdf_e2e_counts`` / ``rdf_e2e_rdf`` (``run()``), ``sq_sums``
(secondary; the raw accumulator of the K identical timed steps over K),
``sq_e2e_ssf`` / ``sq_e2e_wavenumbers`` and ``strong_<cfg>_{counts,rdf,ssf}``.  Every input
is generated from a fixed seed, so two builds run with the same arguments can be compared
output for output.
"""

import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CFG2 = dict(n_ions=20_000, n_frames=2_000, n_bins=201, range=(0.0, 14.5), seed=20260002,
            call_frames=200)
CFG3 = dict(n=500_000, n_frames=1_000, n_bins=100, range=(0.0, 2.5), seed=20260003, ring=32)
CFG4 = dict(n=50_000, n_frames=1_000, n_points=32, n_max=16, seed=20260004, call_frames=125)
CFG5 = dict(n_chains=10_000, chain=100, n_frames=500, n_bins=100, range=(0.0, 2.5),
            n_points=32, n_max=16, seed=20260005, ring=16)
FP64_OPS_PER_PAIR = 21       # DESIGN.md: FP64-pipe instructions per pair evaluation
FP32_OPS_PER_PAIR = 16       # DESIGN.md 4.1b: FP32 instructions per pair of the filter
                             # kernel (3 sub, 3 fma, 3 sub, 3 fma, mul + 2 fma, 1 fma)
FP64_OPS_PER_TERM = 4        # DESIGN.md: DFMA per (q, r) term of the lattice kernel


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--strong", default="cfg4,cfg3,cfg5",
                    help="comma-separated strong-scaling workloads to run")
    ap.add_argument("--strong-reps", type=int, default=5)
    ap.add_argument("--strong-only", action="store_true",
                    help="skip the headline and the secondary; only the strong passes")
    ap.add_argument("--hist", default="auto")
    ap.add_argument("--sq-kernel", default="lattice_dmma",
                    choices=["lattice_dmma", "lattice_fp64"],
                    help="lattice_dmma: FP64 matrix unit (default); lattice_fp64: scalar DFMA")
    ap.add_argument("--arith", default="auto", choices=["auto", "off"],
                    help="auto: fp32 filter + exact fp64 re-evaluation; off: fp64 for "
                         "every pair")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step of every "
                         "measured path computed as DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup < 0:
        ap.error("--warmup must not be negative")
    return a


# ---------------------------------------------------------------------------------
# outputs of the timed paths (--dump-outputs)
# ---------------------------------------------------------------------------------

_OUTPUTS = {}
DUMP_LIMIT_BYTES = 64 << 20


def keep_output(name, array):
    """Records what a timed path returned to its caller in its last step; rank 0 writes."""
    _OUTPUTS[name] = np.array(array, dtype=np.float64)


def dump_outputs(directory):
    """Writes every recorded output as ``directory/<name>.npy``.  The inputs are seeded, so
    two builds run with the same arguments can be compared output for output."""
    total = sum(a.nbytes for a in _OUTPUTS.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT_BYTES}")
    os.makedirs(directory, exist_ok=True)
    for name, a in _OUTPUTS.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_ready(self, timeout=30.0):
        """Blocks until nvidia-smi has printed its first sample: its start-up (NVML /
        driver initialisation, seconds on a fresh box) stalls kernel launches of other
        processes and must not overlap the timed region."""
        t0 = time.time()
        while self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in self.lines:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(pw)), "samples": len(sm),
                "reasons": sorted(reasons)}


def profiled_traffic(kernel_tag, frames_per_launch):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full
    capture (profiles/rNN_<tag>_metrics.csv, newest round first; the capture's frame count
    is in profiles/captures.json, default 20 / 128), scaled to this run's frames per
    launch (the kernel streams every coordinate once, so traffic is linear in frames).
    None if no profile is committed."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    frames_in = {"filter": 20, "pair": 20, "sq": 128}
    try:
        frames_in.update(json.loads((ROOT / "profiles" / "captures.json").read_text()))
    except (OSError, ValueError):
        pass
    for rnd in ("r02", "r01"):
        p = ROOT / "profiles" / f"{rnd}_{kernel_tag}_metrics.csv"
        if not p.exists():
            continue
        tot = 0.0
        try:
            for line in p.read_text().splitlines():
                f = line.split(",")
                if f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(f[2]) * unit[f[1]]
        except (ValueError, KeyError, IndexError):
            continue
        key = f"{rnd}_{kernel_tag}" if f"{rnd}_{kernel_tag}" in frames_in else kernel_tag
        return tot * frames_per_launch / frames_in[key], p.name
    return None, None


def measured_peaks():
    out = {"hbm_gbs": 6650.0, "hbm_source": "fallback (B200_PROFILING.md)",
           "fp64_per_clk_sm": 64.0, "sfu_per_clk_sm": 16.0, "fp32_per_clk_sm": 128.0,
           "fp32_source": "nominal (no profiles/microbench2_r01.json)",
           "pipe_source": "nominal (no profiles/microbench_r01.json)"}
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            out["hbm_gbs"] = float(json.loads(p.read_text())["hbm_gbs"])
            out["hbm_source"] = "MEASURED_PEAKS.json"
        except (ValueError, KeyError):
            pass
    p = ROOT / "profiles" / "microbench_r01.json"
    if p.exists():
        try:
            # GPU-wide instruction rates timed with CUDA events at the 1965 MHz the
            # run held (profiles/microbench_r01_clocks.csv) -> per clock and SM
            mb = json.loads(p.read_text())
            per = 1e9 / (mb["sms"] * mb["clock_khz"] * 1e3)
            out["fp64_per_clk_sm"] = float(mb["dfma"]["gops_per_s"]) * per
            out["sfu_per_clk_sm"] = float(mb["mufu_sin"]["gops_per_s"]) * per
            out["pipe_source"] = "measured: profiles/microbench_r01.json (tools/microbench.cu)"
        except (ValueError, KeyError):
            pass
    p = ROOT / "profiles" / "microbench2_r01.json"
    if p.exists():
        try:
            # FP32 lanes per clock and SM: packed FFMA2 (two lanes per instruction)
            mb = json.loads(p.read_text())
            per = 1e9 / (mb["sms"] * mb["clock_khz"] * 1e3)
            out["fp32_per_clk_sm"] = max(float(mb["ffma"]["gops_per_s"]),
                                         2 * float(mb["ffma2"]["gops_per_s"])) * per
            out["fp32_source"] = "measured: profiles/microbench2_r01.json (tools/microbench2.cu)"
        except (ValueError, KeyError):
            pass
    return out


# ---------------------------------------------------------------------------------
# CPU reference path (restated): oracle distances + real numpy.histogram
# ---------------------------------------------------------------------------------

_CPU_STATE = {}


def _cpu_rdf_frame(f):
    from oracle import reference_port as rp
    u, cat, an = _CPU_STATE["u"]
    ts = u.trajectory[int(f)]
    # mirrors _single_frame_parallel (structure.py:793-835): counts || volume.  method=None:
    # the port chooses brute force / grid search by MDAnalysis' own rule (SURVEY.md
    # Appendix A item 2: grid search from 1e8 pairs up); with r_max = 14.5 in a 29.24 box a
    # grid has two cells per axis, which the restated grid search does not cover -- it then
    # evaluates all pairs, like a two-cell grid would.
    c = rp.radial_histogram(cat.positions, an.positions, CFG2["n_bins"], CFG2["range"],
                            ts.dimensions, method=None)
    return np.concatenate((c, [ts.volume]))


def cpu_rdf(frames, n_jobs):
    """Pairs binned per second by the restated reference path on `n_jobs` processes."""
    import multiprocessing as mp
    t0 = time.perf_counter()
    if n_jobs == 1:
        res = [_cpu_rdf_frame(f) for f in frames]
    else:
        with mp.get_context("fork").Pool(n_jobs) as pool:      # base.py:477-501
            res = pool.map(_cpu_rdf_frame, frames, chunksize=1)
    dt = time.perf_counter() - t0
    tot = np.vstack(res).sum(axis=0)                           # structure.py:842
    return float(tot[:-1].sum()) / dt, dt, tot[:-1].astype(np.int64)


def cpu_sq(coords, wavevectors, n_frames, n_threads):
    from oracle import reference_port as rp
    pos = [coords[f].astype(np.float64) for f in range(n_frames)]
    rp.delta_fourier_transform_sum(wavevectors[:64], pos[0][:1000], n_threads)   # warm-up
    t0 = time.perf_counter()
    for p in pos:
        rho = rp.delta_fourier_transform_sum(wavevectors, p, n_threads)
        _ = (rho * rho.conj()).real
    dt = time.perf_counter() - t0
    return n_frames / dt, dt


def make_cpu_sample(n_frames):
    from mdhelper_b200 import synthetic
    _CPU_STATE["u"] = synthetic.electrolyte(CFG2["n_ions"], n_frames, seed=CFG2["seed"],
                                            pinned=False)


def cfg4_wavevectors():
    """The cfg4 wavevector set (first-octant lattice, |q| <= 2 pi 16 / L) without a GPU."""
    from mdhelper_b200 import synthetic
    L = float(synthetic.box_edge(CFG4["n"], 0.8))
    idx = np.arange(CFG4["n_points"])
    g = 2 * np.pi * idx / np.float32(L)
    ii, jj, kk = np.meshgrid(idx, idx, idx, indexing="ij")
    n = np.stack((jj, ii, kk), axis=-1).reshape(-1, 3)
    wv = np.stack((g[n[:, 0]], g[n[:, 1]], g[n[:, 2]]), axis=-1)
    return wv[np.linalg.norm(wv, axis=1) <= 2 * np.pi * CFG4["n_max"] / L]


# ---------------------------------------------------------------------------------
# reference arm
# ---------------------------------------------------------------------------------

def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import oracle
    from mdhelper_b200 import synthetic
    oracle.build()
    cores = len(os.sched_getaffinity(0))
    fps = cores                                     # one frame per core per step
    n_need = fps * (args.steps + args.warmup)
    make_cpu_sample(min(n_need, 64))
    n_have = len(_CPU_STATE["u"][0].trajectory)
    for s in range(args.warmup):
        cpu_rdf([(s * fps + i) % n_have for i in range(fps)], cores)
    t0 = time.perf_counter()
    binned = 0
    for s in range(args.warmup, args.warmup + args.steps):
        _, _, c = cpu_rdf([(s * fps + i) % n_have for i in range(fps)], cores)
        binned += int(c.sum())
    dt = time.perf_counter() - t0
    keep_output("rdf_counts", c)
    value = binned / dt
    sample = (f"each step = {fps} frames of the workload's 2,000 ({fps * args.steps} in "
              f"all), multiprocessing fork pool of {cores} processes over frames "
              "(mirrors base.py:477-501)")
    # the S(q) half of the metric on the same cores: the restated numba kernel
    # (accelerated.py:124-165, prange over wavevectors) on 3 cfg4 frames
    secondary = None
    if not args.no_secondary:
        pos, _, _ = synthetic.fluid_positions(CFG4["n"], 3, seed=CFG4["seed"], pinned=False)
        wv = cfg4_wavevectors()
        v, dts = cpu_sq(pos, wv, 3, cores)
        secondary = {"metric": "sq_frames_per_s", "value": v, "unit": "frames/s",
                     "config": sq_config(len(wv)),
                     "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores,
                                      "kind": "port",
                                      "sample": f"3 of the workload's 1,000 frames in {dts:.1f} s, "
                                                f"{cores} OpenMP threads over wavevectors"}}
    line = {
        "impl": "reference", "metric": "rdf_pairs_binned_per_s", "value": value,
        "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "secondary": secondary,
        "note": "restated reference CPU path: MDAnalysis is not installable here, so "
                "capped_distance is the C restatement in oracle/ feeding the real "
                "numpy.histogram",
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs)
    emit(line)


def prewarm(step, sync, seconds=0.75):
    """Untimed: run steps until `seconds` of wall time have passed, so the timed
    region starts with the SM clocks already raised."""
    t0 = time.perf_counter()
    s = 0
    while time.perf_counter() - t0 < seconds:
        step(s)
        sync()
        s += 1


def workload_config():
    """Identical in both arms (how a step is batched or sampled is not part of it)."""
    return {"workload": "cfg2: two-group cation-anion partial RDF, 20,000-ion electrolyte "
                        "(10,000 x 10,000 ordered pairs per frame), n_bins=201, "
                        "range=(0, 14.5), L=29.2402, 2,000 synthetic frames per GPU",
            "pairs_per_frame": 100_000_000,
            "cache": "inputs larger than L2: every step streams the 480 MB trajectory "
                     "through the kernels once",
            "parallelism": "frames sharded over GPUs, one all-reduce at the end"}


def sq_config(n_q):
    return {"workload": f"cfg4: direct-sum S(q), N=50,000, n_points=32, q_max=2*pi*16/L -> "
                        f"N_q={n_q}, mode=None, form=exp, fp64, 1,000 synthetic frames per GPU",
            "terms_per_frame": CFG4["n"] * n_q,
            "cache": "inputs larger than L2: every step streams the 600 MB trajectory once"}


# ---------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------

def run_ours(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    cores = len(os.sched_getaffinity(0))

    # ---- CPU baselines first (fork pool before any CUDA context exists) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.strong_only:
        import oracle
        oracle.build()
        make_cpu_sample(2 * cores)
        v1, dt1, _ = cpu_rdf([0], 1)
        vp, dtp, _ = cpu_rdf(list(range(2 * cores)), cores)
        cpu = {"value": vp, "unit": "pairs/s", "cores": cores, "kind": "port",
               "serial_value": v1,
               "sample": f"serial: 1 frame in {dt1:.1f} s; parallel: {2 * cores} frames on a "
                         f"fork pool of {cores} processes in {dtp:.1f} s (same cfg2 frames; "
                         "restated reference path: C capped_distance + numpy.histogram)"}

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from mdhelper_b200 import affinity
    # each rank next to its GPU before any trajectory buffer is allocated
    bound = affinity.bind_to_device(local, world, local) if world > 1 else None

    line = {}
    if not args.strong_only:
        note("headline: cfg2 pair histogram")
        line = bench_rdf(args, rank, world, local, cpu, dist, torch)
        if not args.no_secondary:
            note("secondary: cfg4 structure factor")
            sec = bench_sq(args, rank, world, local, cores, dist, torch)
            if rank == 0:
                line["secondary"] = sec
    if not args.no_strong:
        strong = {}
        for which in [w for w in args.strong.split(",") if w]:
            note(f"strong scaling pass: {which}")
            res = bench_strong(which, args, rank, world, local, dist, torch)
            if rank == 0:
                strong[which] = res
        if rank == 0:
            line["strong"] = strong
    if rank == 0:
        if args.strong_only:
            line = dict({"metric": "strong_scaling_passes", "n_gpus": world}, **line)
        if bound is not None:
            line["affinity"] = bound
        if args.dump_outputs:
            dump_outputs(args.dump_outputs)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def bench_rdf(args, rank, world, local, cpu, dist, torch):
    from mdhelper_b200 import _lib, synthetic
    from mdhelper_b200.analysis._binning import squared_thresholds
    from mdhelper_b200.analysis.structure import RadialDistributionFunction
    from mdhelper_b200.universe import SyntheticUniverse

    K, W, cf = args.steps, args.warmup, CFG2["call_frames"]
    n_frames = CFG2["n_frames"]
    u, cat, an = synthetic.electrolyte(CFG2["n_ions"], n_frames, seed=CFG2["seed"] + 1000 * rank)
    n1, n2, N = cat.n_atoms, an.n_atoms, CFG2["n_ions"]
    coords = u.trajectory.coordinates
    boxes = np.ascontiguousarray(u.trajectory.unitcells[:, :3])

    # ---- value: coordinates resident in HBM ----
    dev = torch.from_numpy(coords).cuda(non_blocking=True)
    torch.cuda.synchronize()
    ctx = _lib.Context(local)
    thr = squared_thresholds(CFG2["n_bins"], CFG2["range"])
    ctx.rdf_set_filter(args.arith)
    ctx.rdf_configure(n1, n2, False, thr, *CFG2["range"], hist=args.hist)
    base = dev.data_ptr()

    def call(f0):
        nf = min(cf, n_frames - f0)
        ctx.rdf_accumulate(base + 4 * 3 * N * f0, 3 * N, base + 4 * 3 * (N * f0 + n1), 3 * N,
                           boxes[f0:f0 + nf], nf, device=True)
        return nf

    def step(_s):
        return sum(call(f0) for f0 in range(0, n_frames, cf))

    # the clock sampler starts first: nvidia-smi's own start-up (NVML init) must be
    # over before the timed region; only samples inside [wall0, wall1] are used
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_ready()
    if world > 1:
        dist.barrier()
    prewarm(lambda s: call((s * cf) % n_frames), ctx.sync, 1.5)   # clocks up (untimed)
    for s in range(W):
        step(s)
    # the tail of the timed region once, untimed: the first fetch -> device copy ->
    # all-reduce of a process pays one-off initialisation (tens of ms on a fresh box)
    warm = torch.from_numpy(ctx.rdf_fetch()).cuda()
    if world > 1:
        dist.all_reduce(warm)
    torch.cuda.synchronize()
    ctx.sync()
    ctx.rdf_reset()
    ctx.kernel_time(reset=True)
    launches0 = ctx.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    ev0.record()
    frames_done = 0
    for s in range(W, W + K):
        frames_done += step(s)
    counts = torch.from_numpy(ctx.rdf_fetch()).cuda()
    if world > 1:
        dist.all_reduce(counts)
    ev1.record()
    torch.cuda.synchronize()
    wall1 = time.time()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    launches = ctx.launch_count() - launches0
    binned_total = int(counts.sum().item())
    # every timed step bins the same frames, so the integer counts of the timed region are
    # exactly K times those of its last step
    total = counts.cpu().numpy()
    assert not (total % K).any(), "timed steps binned different counts"
    keep_output("rdf_counts", total // K)
    evals_local = ctx.rdf_pair_evaluations()
    fstats = ctx.rdf_filter_stats()
    filtered = bool(fstats["eligible"]) and args.arith != "off" and args.hist in ("auto", "warp_atomic")
    # per-launch duration of the pair kernel: CUDA events recorded around every
    # launch of the timed region, on the launching stream (mdh_kernel_time)
    kern_total_ms, kern_calls, _, _ = ctx.kernel_time(reset=True)
    kern_ms = kern_total_ms / max(kern_calls, 1)
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    value = binned_total / (ms * 1e-3)
    del dev
    ctx.close()

    note("headline: end to end through run()")
    # ---- e2e: public class, pinned host memory, H2D + D2H inside the timed region ----
    # weak scaling like `value`: run() shards the frames it is given over the ranks
    # (np.array_split), so every rank exposes a trajectory of world * 2,000 frames whose
    # own share is its 2,000 local frames, and the counts come back summed over the ranks
    ue = SyntheticUniverse(coords, u.trajectory.unitcells[0], n_frames=world * n_frames)
    cat_e, an_e = ue.select(slice(0, n1)), ue.select(slice(n1, N))
    rdf = RadialDistributionFunction(cat_e, an_e, n_bins=CFG2["n_bins"], range=CFG2["range"],
                                     verbose=False, batch_frames=cf, hist=args.hist,
                                     arith=args.arith)
    for s in range(max(1, min(W, 2))):
        rdf.run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_binned = 0
    for s in range(K):
        rdf.run()
        e2e_binned += int(rdf.results.counts.sum())       # already summed over ranks
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = e2e_binned / float(e2e_s.item())
    keep_output("rdf_e2e_counts", rdf.results.counts)
    keep_output("rdf_e2e_rdf", rdf.results.rdf)
    if rank != 0:
        return None

    peaks = measured_peaks()
    sm_mhz = clocks["sm_mhz"] or clocks.get("sm_max_mhz") or 1965.0
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    fp64_peak = peaks["fp64_per_clk_sm"] * n_sm * sm_mhz * 1e6        # instr/s
    fp32_peak = peaks["fp32_per_clk_sm"] * n_sm * sm_mhz * 1e6        # FP32 lanes/s
    evals_per_launch = cf * n1 * n2
    alg_bytes = cf * (n1 + n2) * 16 + CFG2["n_bins"] * 8            # float4 in, counts out
    hbm = {"achieved_gbs": alg_bytes / (kern_ms * 1e-3) / 1e9,
           "peak_gbs": peaks["hbm_gbs"], "source": peaks["hbm_source"],
           "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    fp64_equiv = evals_per_launch * FP64_OPS_PER_PAIR / (kern_ms * 1e-3)
    if filtered:
        # the kernel that runs: fp32 filter (packed FFMA2/FADD2 on the FP32 pipe);
        # about 1 pair in 1,500 is re-evaluated in fp64 (counted in fstats)
        achieved = evals_per_launch * FP32_OPS_PER_PAIR / (kern_ms * 1e-3)
        traffic, tfile = profiled_traffic("filter", cf)
        roofline = {
            "kernel": "rdf_filter_kernel", "bound": "fp32_pipe",
            "achieved": achieved / 1e9, "peak": fp32_peak / 1e9, "unit": "Ginstr/s",
            "frac": achieved / fp32_peak,
            "traffic": traffic,
            "traffic_note": f"dram__bytes_read+write of profiles/{tfile} scaled to this "
                            "launch's frames; bytes",
            "per_unit": f"{FP32_OPS_PER_PAIR} FP32 operations per pair evaluation "
                        "(minimum image, squared distance, bin coordinate; issued as "
                        "packed f32x2 instructions)",
            "units_per_launch": evals_per_launch, "launch_ms": kern_ms,
            "peak_source": f"{peaks['fp32_source']}; {peaks['fp32_per_clk_sm']:.1f} FP32 "
                           f"lanes/clk/SM x {n_sm} SMs x {sm_mhz:.0f} MHz (sampled)",
            "fp64_pipe_equivalent_frac": fp64_equiv / fp64_peak,
            "fp64_pipe_equivalent_note": "the same pair rate expressed against the bound "
                                         "of a kernel that evaluates the reference's 21 "
                                         "FP64 instructions for every pair (the --arith "
                                         "off kernel reaches 0.62 of it)",
            "filter": {"deferred_entries": fstats["deferred_entries"],
                       "inline_entries": fstats["inline_entries"],
                       "declined_frames": fstats["declined_frames"]},
            "hbm": hbm,
        }
    else:
        traffic, tfile = profiled_traffic("pair", cf)
        roofline = {
            "kernel": "rdf_allpairs_kernel", "bound": "fp64_pipe",
            "achieved": fp64_equiv / 1e9, "peak": fp64_peak / 1e9, "unit": "Ginstr/s",
            "frac": fp64_equiv / fp64_peak,
            "traffic": traffic,
            "traffic_note": f"dram__bytes_read+write of profiles/{tfile} scaled to this "
                            "launch's frames; bytes",
            "per_unit": f"{FP64_OPS_PER_PAIR} FP64-pipe instructions per pair evaluation "
                        "(no FMA fusion allowed)",
            "units_per_launch": evals_per_launch, "launch_ms": kern_ms,
            "peak_source": f"{peaks['pipe_source']}; {peaks['fp64_per_clk_sm']:.1f} "
                           f"instr/clk/SM x {n_sm} SMs x {sm_mhz:.0f} MHz (sampled)",
            "hbm": hbm,
        }
    return {
        "metric": "rdf_pairs_binned_per_s", "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(),
        "step": f"one pass over the 2,000 frames: {n_frames // cf} C-ABI calls of {cf} frames",
        "pairs_evaluated_per_s": evals_local * world / (ms * 1e-3),
        "frames_per_s": frames_done * world / (ms * 1e-3),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "pairs/s",
                "h2d_bytes_per_step": world * (n_frames * (n1 + n2) * 12 + n_frames * 48),
                "d2h_bytes_per_step": world * CFG2["n_bins"] * 8,
                "api": "RadialDistributionFunction(cations, anions, n_bins=201, "
                       "range=(0, 14.5)).run() over the 2,000 frames per step"},
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
    }


def bench_sq(args, rank, world, local, cores, dist, torch):
    """S(q) frames/s for cfg4 (N=50,000, N_q=2,446, 1,000 frames per GPU), device-resident
    and end to end; step = one pass over the 1,000 frames."""
    from mdhelper_b200 import _lib, synthetic
    from mdhelper_b200.analysis.structure import StructureFactor
    from mdhelper_b200.universe import SyntheticUniverse
    K, W, cf = args.steps, args.warmup, CFG4["call_frames"]
    n_frames = CFG4["n_frames"]
    u = synthetic.lj_fluid(CFG4["n"], n_frames, seed=CFG4["seed"] + 1000 * rank)
    coords = u.trajectory.coordinates
    L = float(u.trajectory.unitcells[0, 0])
    q_max = 2 * np.pi * CFG4["n_max"] / L
    ue = SyntheticUniverse(coords, u.trajectory.unitcells[0], n_frames=world * n_frames)
    sf = StructureFactor([ue.atoms], n_points=CFG4["n_points"], q_max=q_max, verbose=False,
                         batch_frames=cf, kernel=args.sq_kernel)
    dmma = args.sq_kernel == "lattice_dmma"
    n_q = len(sf._wavenumbers)
    N = CFG4["n"]

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v1, dt1 = cpu_sq(coords, sf._wavevectors, 1, 1)
        vp, dtp = cpu_sq(coords, sf._wavevectors, 3, cores)
        cpu = {"value": vp, "unit": "frames/s", "cores": cores, "kind": "port",
               "serial_value": v1,
               "sample": f"serial: 1 frame in {dt1:.1f} s; {cores} OpenMP threads over "
                         f"wavevectors: 3 frames in {dtp:.1f} s (C restatement of "
                         "accelerated.py:81-165)"}

    dev = torch.from_numpy(coords).cuda()
    ctx = _lib.Context(local)
    ctx.sq_configure(N, [0, N], sf._wavevectors, [(-1, -1)], lattice_n=sf._lattice_n,
                     lattice_b=sf._lattice_b, mode=args.sq_kernel)
    assert ctx.sq_kernel() == args.sq_kernel, ctx.sq_kernel()
    tiling = ctx.sq_tiling()
    base = dev.data_ptr()

    def call(f0):
        nf = min(cf, n_frames - f0)
        ctx.sq_accumulate(base + 4 * 3 * N * f0, 3 * N, nf, device=True)
        return nf

    def step(_s):
        return sum(call(f0) for f0 in range(0, n_frames, cf))

    prewarm(lambda s: call((s * cf) % n_frames), ctx.sync, 0.4)
    for s in range(W):
        step(s)
    warm = torch.from_numpy(ctx.sq_fetch()).cuda()
    if world > 1:
        dist.all_reduce(warm)
    torch.cuda.synchronize()
    ctx.sync()
    ctx.sq_reset()
    ctx.kernel_time(reset=True)
    l0 = ctx.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    frames = 0
    for s in range(W, W + K):
        frames += step(s)
    acc = torch.from_numpy(ctx.sq_fetch()).cuda()
    if world > 1:
        dist.all_reduce(acc)
    ev1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    launches = ctx.launch_count() - l0
    # raw fp64 sums of the K identical timed steps: their mean is the last step's sums to
    # rounding
    keep_output("sq_sums", acc.cpu().numpy() / K)
    _, _, kern_total_ms, kern_calls = ctx.kernel_time(reset=True)
    kern_ms = kern_total_ms / max(kern_calls, 1)
    del dev
    ctx.close()

    note("secondary: end to end through run()")
    for s in range(max(1, min(W, 2))):
        sf.run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_frames = 0
    for s in range(K):
        sf.run()
        e2e_frames += sf.n_frames                 # all ranks together
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    keep_output("sq_e2e_ssf", sf.results.ssf)
    keep_output("sq_e2e_wavenumbers", sf.results.wavenumbers)
    if rank != 0:
        return None

    peaks = measured_peaks()
    n_sm = torch.cuda.get_device_properties(local).multi_processor_count
    terms = cf * N * n_q
    achieved = terms * FP64_OPS_PER_TERM / (kern_ms * 1e-3)
    peak = peaks["fp64_per_clk_sm"] * n_sm * 1965e6
    traffic, tfile = profiled_traffic("sq", cf)
    return {
        "metric": "sq_frames_per_s", "value": frames * world / (ms * 1e-3), "unit": "frames/s",
        "config": sq_config(n_q),
        "step": f"one pass over the 1,000 frames: {n_frames // cf} C-ABI calls of {cf} frames",
        "ms_per_step": ms / K, "gpu_launches": launches,
        "e2e": {"value": e2e_frames / float(e2e_s.item()), "unit": "frames/s",
                "h2d_bytes_per_step": world * n_frames * N * 12,
                "d2h_bytes_per_step": world * n_q * 8,
                "api": "StructureFactor([atoms], n_points=32, q_max=...).run() over the "
                       "1,000 frames per step"},
        # the DMMA kernel runs on the FP64 matrix unit: the contract's "tensor" bound, in
        # TFLOP/s (2 flop per FMA); the scalar kernel is bound by the FP64 FMA pipe
        "roofline": {"kernel": "sq_lattice_mma_kernel" if dmma else "sq_lattice_kernel<double>",
                     "bound": "tensor" if dmma else "fp64_pipe",
                     "achieved": achieved * 2 / 1e12 if dmma else achieved / 1e9,
                     "peak": peak * 2 / 1e12 if dmma else peak / 1e9,
                     "unit": "TFLOP/s" if dmma else "Ginstr/s",
                     "frac": achieved / peak,
                     "bound_note": ("fp64 matrix unit (mma.m8n8k4.f64 = SASS DMMA.8x8x4); "
                                    "algorithmic work = 4 fp64 FMA = 8 flop per (q, r) term")
                     if dmma else None,
                     "traffic": traffic,
                     "traffic_note": f"dram__bytes_read+write of profiles/{tfile} scaled to "
                                     "this launch's frames; bytes",
                     "nominal_vs_reachable":
                         ("DMMA.8x8x4 sustains the nominal 63.6 FMA/clk/SM "
                          "(profiles/microbench3_r01.json); the (column group x nz tile) "
                          "tiling of the |q| <= q_max sphere carries padding slots that "
                          "are executed but not counted as algorithmic work") if dmma else
                         ("a DFMA with three register operands sustains 42.6/clk/SM "
                          "(profiles/microbench2_r01.json), 0.67 of the nominal rate used "
                          "as peak"),
                     "per_unit": f"{FP64_OPS_PER_TERM} fp64 FMA per (q, r) term (complex "
                                 "multiply-accumulate)" + (", issued as DMMA m8n8k4 "
                                 "(256 FMA per warp instruction)" if dmma else ""),
                     "units_per_launch": terms, "launch_ms": kern_ms,
                     "tiling": (dict(tiling, executed_over_algorithmic=tiling["tiles"] * 64 / n_q,
                                     note="(column group x nz tile) pairs of 64 accumulator "
                                          "slots; the DMMAs of padding slots are executed but "
                                          "not counted in `achieved`") if dmma else None),
                     "peak_source": f"{peaks['pipe_source']}; {peaks['fp64_per_clk_sm']:.1f} "
                                    f"instr/clk/SM x {n_sm} SMs x 1965 MHz (max clock)",
                     "sfu_equivalent_frac": (terms * 2 / (kern_ms * 1e-3))
                     / (peaks["sfu_per_clk_sm"] * n_sm * 1965e6)},
        "cpu_baseline": cpu,
    }


# ---------------------------------------------------------------------------------
# strong scaling: the named configurations at their named scale
# ---------------------------------------------------------------------------------

def bench_strong(which, args, rank, world, local, dist, torch):
    """One named configuration, a FIXED frame list split over the ranks, through the public
    classes from host memory.  Every rank builds the same seeded ring of distinct frames
    (SURVEY.md section 8(d): a ring may be cycled to bound host memory) and analyses its
    block of the frame list (np.array_split, as base.py:433-441); afterwards rank 0
    recomputes the whole list alone and compares."""
    from mdhelper_b200 import synthetic
    from mdhelper_b200.analysis import CombinedAnalysis
    from mdhelper_b200.analysis.base import single_rank
    from mdhelper_b200.analysis.structure import RadialDistributionFunction, StructureFactor
    from mdhelper_b200.universe import SyntheticUniverse

    def ring_universe(pos, L, n_frames, **kw):
        return SyntheticUniverse(pos, np.array([L, L, L, 90, 90, 90], np.float32),
                                 n_frames=n_frames, **kw)

    rdf = sf = None
    if which == "cfg4":
        ring = 250
        pos, L, keep = synthetic.fluid_positions(CFG4["n"], ring, seed=CFG4["seed"])
        n_frames, n_part = CFG4["n_frames"], CFG4["n"]
        u = ring_universe(pos, L, n_frames)
        sf = StructureFactor([u.atoms], n_points=CFG4["n_points"],
                             q_max=2 * np.pi * CFG4["n_max"] / float(L), verbose=False,
                             kernel=args.sq_kernel)
        name = ("cfg4: direct-sum S(q), 50,000 particles, N_q=2,446, 1,000 frames "
                f"(ring of {ring} distinct frames)")
    elif which == "cfg3":
        ring = CFG3["ring"]
        pos, L, keep = synthetic.fluid_positions(CFG3["n"], ring, seed=CFG3["seed"])
        n_frames, n_part = CFG3["n_frames"], CFG3["n"]
        u = ring_universe(pos, L, n_frames)
        rdf = RadialDistributionFunction(u.atoms, n_bins=CFG3["n_bins"], range=CFG3["range"],
                                         verbose=False, arith=args.arith)
        name = ("cfg3: RDF with cut-off 2.5 (cell list), 500,000-particle LJ fluid, 1,000 "
                f"frames (ring of {ring} distinct frames)")
    elif which == "cfg5":
        ring = CFG5["ring"]
        um = synthetic.polymer_melt(CFG5["n_chains"], CFG5["chain"], ring, seed=CFG5["seed"])
        pos, L = um.trajectory.coordinates, um.trajectory.unitcells[0, 0]
        keep = um
        n_frames, n_part = CFG5["n_frames"], CFG5["n_chains"] * CFG5["chain"]
        chain = np.repeat(np.arange(CFG5["n_chains"]), CFG5["chain"])
        u = ring_universe(pos, L, n_frames, resindices=chain, segindices=chain)
        rdf = RadialDistributionFunction(u.atoms, n_bins=CFG5["n_bins"], range=CFG5["range"],
                                         verbose=False, arith=args.arith)
        sf = StructureFactor([u.atoms], n_points=CFG5["n_points"],
                             q_max=2 * np.pi * CFG5["n_max"] / float(L), verbose=False,
                             kernel=args.sq_kernel)
        name = ("cfg5: combined RDF (cut-off 2.5) + S(q) (N_q=2,446) pass, 1,000,000-bead "
                f"polymer melt, 500 frames (ring of {ring} distinct frames)")
    else:
        raise SystemExit(f"unknown strong workload {which}")

    job = CombinedAnalysis(rdf, sf) if (rdf is not None and sf is not None) else (rdf or sf)

    def one_pass():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        job.run()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return float(dt.item())

    one_pass()                                     # allocations, configuration, clocks
    one_pass()                                     # the staging plan has the first pass's rates
    for a in (rdf, sf):
        if a is not None:
            a._ctx.kernel_time(reset=True)
    times = [one_pass() for _ in range(max(1, args.strong_reps))]
    best, mean = min(times), float(np.mean(times))
    kern = {}
    if rdf is not None:
        kern["rdf_kernel_ms_rank0"] = rdf._ctx.kernel_time()[0] / len(times)
        kern["rdf_pair_evaluations_rank0"] = rdf._pair_evaluations
    if sf is not None:
        kern["sq_kernel_ms_rank0"] = sf._ctx.kernel_time()[2] / len(times)
    out = {"workload": name, "n_gpus": world, "frames": n_frames, "scaling": "strong",
           "passes_timed": len(times), "e2e_s_mean": mean, "e2e_s_best": best,
           "e2e_s_passes": [round(t, 6) for t in times],
           "frames_per_s": n_frames / mean,
           "h2d_bytes_per_pass": n_frames * n_part * 12,
           "api": ("CombinedAnalysis(rdf, ssf).run()" if isinstance(job, CombinedAnalysis)
                   else type(job).__name__ + "(...).run()") + " over the whole frame list, "
                  "host memory -> results"}
    if rdf is not None:
        counts = rdf.results.counts.copy()
        out["pairs_binned_per_s"] = float(counts.sum()) / mean
        out["counts_sum"] = int(counts.sum())
        keep_output(f"strong_{which}_counts", counts)
        keep_output(f"strong_{which}_rdf", rdf.results.rdf)
    if sf is not None:
        ssf = sf.results.ssf.copy()
        keep_output(f"strong_{which}_ssf", ssf)
    # ---- multi-GPU parity: rank 0 alone over the whole frame list ----
    if world > 1:
        ok = torch.ones(1, device="cuda")
        if rank == 0:
            with single_rank():
                job.run()
            good = True
            if rdf is not None:
                good = good and bool(np.array_equal(rdf.results.counts, counts))
                out["parity_counts_equal"] = bool(np.array_equal(rdf.results.counts, counts))
            if sf is not None:
                rel = float(np.max(np.abs(sf.results.ssf - ssf)
                                   / np.maximum(np.abs(sf.results.ssf), 1e-300)))
                out["parity_ssf_max_rel"] = rel
                good = good and rel <= 1e-12
            out["multi_gpu_parity"] = good
            ok[0] = 1.0 if good else 0.0
        dist.broadcast(ok, 0)
        if float(ok.item()) != 1.0 and rank == 0:
            # reported, not fatal: the line still carries every other measurement
            print(f"multi-GPU parity FAILED for {which}: {out}", file=sys.stderr)
    else:
        out["multi_gpu_parity"] = None           # one rank: nothing to compare
    out.update(kern)
    del job, rdf, sf, u, keep
    torch.cuda.empty_cache()
    return out if rank == 0 else None


_T0 = time.time()


def note(msg: str) -> None:
    """Progress on stderr (rank 0): which part is running, seconds since start."""
    if int(os.environ.get("RANK", 0)) == 0:
        print(f"[bench {time.time() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the real stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    # Libraries print to stdout behind our back (NCCL: "NCCL version ..." at communicator
    # creation): everything but the result line goes to stderr.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    # a run that stalls says where: stack traces of all threads on stderr every 5 minutes
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("MDH_BENCH_STALL_S", 300)),
                                      repeat=True, file=sys.stderr)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
