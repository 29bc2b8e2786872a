"""Cost of a mixed sensor table: the C2 shape (1024 scenes, ~200 points per frame, 3-D pose net), serial mode, per-step
CUDA events on the library's stream with L2 flushed before every timed step, as bench.py's `value` is taken.

Two contexts, stepped alternately in blocks of --block frames:
  untouched  the table as mmw_create filled it (one mounting, one radar profile): bench.py's workload
  mixed      4 mountings x 2 radar profiles, scene s generated as seen from its own sensor
Prints ms per step for each, the per-kernel times of step_kernel, dbscan_big_kernel and pose_feature_kernel, and the
GPU's name and power limit.  Run from the repository root: python profiles/scene_sensors.py
"""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from mmwave_msc_b200 import pose_weights as pw, synth  # noqa: E402
from mmwave_msc_b200.batched import BatchedTracker, default_config  # noqa: E402

MOUNTS = [(1.2, -15.0, 2.2), (1.8, -5.0, 2.5), (2.4, 0.0, 3.0), (1.8, 5.0, 2.5)]     # s_height, s_tilt_deg, z_max
PROFILES = [0.0626, 0.125]
DEFAULT_RES = 0.0626


def frames(S, n, mixed):
    """Per frame (rows with the Doppler index, offsets, dt) on the device; scene s's sensor."""
    out = [[] for _ in range(n)]
    dts = np.zeros((n, S))
    for s in range(S):
        h, t, _ = MOUNTS[s % 4] if mixed else (synth.S_HEIGHT, synth.S_TILT_DEG, None)
        res = PROFILES[(s // 4) % 2] if mixed else DEFAULT_RES
        sc = synth.gen_scene(s, n, synth.SceneSpec(s_height=h, s_tilt_deg=t, doppler_res=res))
        dts[:, s] = sc.dts()
        for f, fr in enumerate(sc.frames):
            r = fr.copy()
            r[:, 3] = np.rint(fr[:, 3].astype(np.float64) / res)
            out[f].append(r)
    dev = []
    for f in range(n):
        off = np.zeros(S + 1, np.int32)
        off[1:] = np.cumsum([len(r) for r in out[f]])
        dev.append((torch.from_numpy(np.concatenate(out[f])).cuda(), torch.from_numpy(off).cuda(),
                    torch.from_numpy(dts[f].copy()).cuda()))
    return dev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=40, help="timed steps per context")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--block", type=int, default=5, help="steps per context between switches")
    args = ap.parse_args()
    S, K, W = args.scenes, args.steps, args.warmup
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    weights = pw.make_pose_weights(pw.VARIANT_3D)
    arms = {}
    for name, mixed in (("untouched", False), ("mixed", True)):
        bt = BatchedTracker(S, max_points=256, max_tracks=8, config=default_config(doppler_res=DEFAULT_RES))
        bt.load_pose_weights(weights)
        if mixed:
            bt.set_scene_sensors(s_height=[MOUNTS[s % 4][0] for s in range(S)],
                                 s_tilt_deg=[MOUNTS[s % 4][1] for s in range(S)],
                                 z_max=[MOUNTS[s % 4][2] for s in range(S)],
                                 doppler_res=[PROFILES[(s // 4) % 2] for s in range(S)])
        arms[name] = {"bt": bt, "dev": frames(S, W + 2 * K, mixed), "f": 0, "ms": []}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def step(a):
        p, o, d = a["dev"][a["f"]]
        a["bt"].step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True)
        a["f"] += 1

    for a in arms.values():
        for _ in range(W):
            step(a)
        a["bt"].sync()
    for b0 in range(0, K, args.block):
        for a in arms.values():
            stream = torch.cuda.ExternalStream(a["bt"].stream)
            ev = []
            for _ in range(b0, min(K, b0 + args.block)):
                with torch.cuda.stream(stream):
                    flush.fill_(a["f"] & 0xff)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                step(a)
                e1.record(stream)
                ev.append((e0, e1))
            a["bt"].sync()
            a["ms"] += [x.elapsed_time(y) for x, y in ev]
    print("GPU: %s" % gpu)
    print("C2 shape: %d scenes, serial mode with pose, L2 flushed before every timed step, %d steps per arm" % (S, K))
    for name, a in arms.items():
        ms = np.array(a["ms"])
        kern = a["bt"].profile_kernels(lambda i, a=a: step(a), K)
        print("%-9s  %.4f ms/step (median %.4f, min %.4f)   step %.4f  dbscan_big %.4f  pose_features %.4f ms"
              % (name, ms.mean(), np.median(ms), ms.min(), kern.get("step", 0.0), kern.get("dbscan_big", 0.0),
                 kern.get("pose_features", 0.0)))


if __name__ == "__main__":
    main()
