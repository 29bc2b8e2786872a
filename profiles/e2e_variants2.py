#!/usr/bin/env python
"""What separates the end-to-end loop (mmw_run_frames on pinned host buffers) from the device-resident throughput mode:
one variant per process (environment knobs are read once).  VARIANT = resident | resident_serial | full | compact | compact_serial | full_serial"""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from mmwave_msc_b200 import _lib, pose_weights as pw, synth  # noqa: E402
from mmwave_msc_b200.batched import BatchedTracker, default_config  # noqa: E402

variant = os.environ.get("VARIANT", "compact")
S, PRIME, K, REPS = 1024, 12, 40, 3
batches = synth.gen_batch(range(S), PRIME + (REPS + 1) * K)
f32, i16 = zip(*[bench.lattice_rows(b.points) for b in batches])
bt = BatchedTracker(S, config=default_config(doppler_res=bench.DOPPLER_RES, xyz_q_format=9))
bt.load_pose_weights(pw.make_pose_weights(pw.VARIANT_3D))
n = S * 8 * _lib.RESULT_FLOATS
for f in range(PRIME):
    bt.step(f32[f], batches[f].offsets, batches[f].dt, pose=True)
bt.sync()


def pin(a):
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


lo, hi = PRIME, PRIME + (REPS + 1) * K
R = pin(np.concatenate(i16[lo:hi] + (i16[hi - 1],) * 4))
fro = np.cumsum([0] + [len(r) for r in i16[lo:hi]]).astype(np.int64)
O = pin(np.stack([b.offsets for b in batches[lo:hi]]))
D = pin(np.stack([b.dt for b in batches[lo:hi]]))
res = pin(np.zeros((hi - lo + 4, n), np.float32))
cnt = pin(np.zeros(hi - lo + 4, np.int32))
dev = [(torch.from_numpy(f32[f]).cuda(), torch.from_numpy(batches[f].offsets).cuda(), torch.from_numpy(batches[f].dt).cuda())
       for f in range(lo, hi)] if variant.startswith("resident") else None
stream = torch.cuda.ExternalStream(bt.stream, device=0)
rd = torch.empty(n, dtype=torch.float32, device="cuda")
out = []
for rep in range(REPS + 1):
    a, b = rep * K, (rep + 1) * K
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if variant.startswith("resident"):
        for p, o, d in dev[a:b]:
            bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=not variant.endswith("_serial"))
        bt.pack_results(rd.data_ptr())
        bt.sync()
    else:
        blk = (R[fro[a]:fro[b]], (fro[a:b + 1] - fro[a]).astype(np.int64), O[a:b], D[a:b], res[a:b])
        bt.run_frames(*blk, n_records=cnt[a:b] if variant.startswith("compact") else None,
                      pipeline=not variant.endswith("_serial"))
    torch.cuda.synchronize()
    out.append((time.perf_counter() - t0) / K * 1e6)
print("%-10s : us per frame %s (first = warm-up)" % (variant, [round(v) for v in out]))
