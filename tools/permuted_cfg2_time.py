"""cfg2 frames (bench.py's headline workload) with both groups randomly permuted in every
frame: time per 200-frame rdf_accumulate call on device-resident coordinates (CUDA events
over 10 passes of 400 frames), the filter statistics and a checksum of the counts.

Shows that the all-pairs filter's x-sorted tiles do not depend on the generator's lattice
order.  Runs against the package of the current directory:
    python tools/permuted_cfg2_time.py"""
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.getcwd())
from mdhelper_b200 import _lib, synthetic
from mdhelper_b200.analysis._binning import squared_thresholds
NF, CF = 400, 200
u, cat, an = synthetic.electrolyte(20_000, NF, seed=20260002)
c = np.array(u.trajectory.coordinates[:NF], np.float32)
n1 = cat.n_atoms
rng = np.random.default_rng(1)
for f in range(NF):
    c[f, :n1] = c[f, rng.permutation(n1)]
    c[f, n1:] = c[f, n1 + rng.permutation(20_000 - n1)]
boxes = np.ascontiguousarray(u.trajectory.unitcells[:NF, :3])
dev = torch.from_numpy(c).cuda()
base = dev.data_ptr(); N = 20_000
ctx = _lib.Context(0)
ctx.rdf_configure(n1, N - n1, False, squared_thresholds(201, (0.0, 14.5)), 0.0, 14.5)
def step():
    for f0 in range(0, NF, CF):
        ctx.rdf_accumulate(base + 4 * 3 * N * f0, 3 * N, base + 4 * 3 * (N * f0 + n1), 3 * N,
                           boxes[f0:f0 + CF], CF, device=True)
for _ in range(3): step()
ctx.sync(); ctx.rdf_reset()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
K = 10
e0.record()
for _ in range(K): step()
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / (K * NF / CF)
st = ctx.rdf_filter_stats()
counts = ctx.rdf_fetch()
print(json.dumps({"ms_per_200_frames": ms, "stats": st, "binned": int(counts.sum()),
                  "checksum": int((counts * np.arange(1, 202)).sum())}))
ctx.close()
