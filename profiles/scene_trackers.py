"""Cost of the per-scene tracker table (mmw_set_scene_trackers) and what one context with a mixed table gives.

Prints, with the GPU's name and power limit read in the same run:
  - the mmw_profile times (CUDA events around every launch) of step_kernel and dbscan_big_kernel at the C2 shape (1024
    scenes, 256 points per frame, 8 tracks, 3-D pose net, serial steps); --kernels-only stops here, so that the same
    numbers can be taken from another build (MMW_LIB=path/to/libmmw.so);
  - the wall time of one mmw_set_scene_trackers call (host clock around the call and mmw_sync) for 1 scene and for all
    1024, with and without a change of the DBSCAN constants (which queues the histogram-flag kernel), median of --reps;
  - 1024 dense scenes (C3 input: 1000 points per frame, 10 targets) at max_points = 1024, max_tracks = 16, half tuned as
    C2 (tr_max_tracks = 4) and half as C3 (tr_max_tracks = 10): one context with a mixed table against the two halves
    in two contexts stepped back to back.  Wall time per frame (host clock around the steps and the synchronisation of
    both contexts), median over --steps frames after --warmup frames.  Reported, not a target.
Run from the repository root: python profiles/scene_trackers.py
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from mmwave_msc_b200 import pose_weights as pw, synth  # noqa: E402
from mmwave_msc_b200.batched import BatchedTracker, default_config  # noqa: E402


def wall(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def device_frames(batches, lo, hi, tile=1):
    """Per frame (points, offsets, dt) on the device of scenes lo .. hi - 1 of the batches, the whole set tiled."""
    out = []
    for b in batches:
        pts = [b.points[b.offsets[lo]:b.offsets[hi]]] * tile
        cnt = np.tile(np.diff(b.offsets[lo:hi + 1]), tile)
        off = np.zeros(cnt.size + 1, np.int32)
        off[1:] = np.cumsum(cnt)
        dt = np.tile(b.dt[lo:hi], tile)
        out.append((torch.from_numpy(np.ascontiguousarray(np.concatenate(pts))).cuda(), torch.from_numpy(off).cuda(),
                    torch.from_numpy(dt).cuda()))
    return out


def step(bt, fr):
    p, o, d = fr
    bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--warmup", type=int, default=15)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--kernels-only", action="store_true")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("GPU: %s" % gpu)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    S = 1024
    n_fr = args.warmup + args.steps
    bt = BatchedTracker(S, max_points=256, max_tracks=8)
    bt.load_pose_weights(W)
    c2 = device_frames(synth.gen_batch(range(S), n_fr), 0, S)
    for f in range(args.warmup):
        step(bt, c2[f])
    k = bt.profile_kernels(lambda i: step(bt, c2[args.warmup + i]), args.steps)
    print("C2 shape, serial steps %d..%d, mmw_profile ms per launch: step %.4f, dbscan_big %.4f"
          % (args.warmup, n_fr - 1, k["step"], k["dbscan_big"]))
    if args.kernels_only:
        return

    lib, h = bt.lib, bt._h
    tab = bt.scene_trackers()
    other = tab.copy()
    other["tr_gate"] = 5.0
    dbs = tab.copy()
    dbs["db_eps"] = 0.31
    print("mmw_set_scene_trackers + mmw_sync, wall ms, median of %d (host clock); the context is idle" % args.reps)
    for n in (1, S):
        for name, new in (("tracker field", other), ("DBSCAN field", dbs)):
            flip = [new, tab]
            i = [0]

            def call():
                lib.mmw_set_scene_trackers(h, 0, n, flip[i[0] & 1].ctypes.data)
                i[0] += 1
                bt.sync()

            call()
            print("  %4d scene(s), %-13s changed: %.4f ms" % (n, name, wall(call, args.reps)))
    bt.close()

    # the mixed fleet: half C2 tuning, half C3 tuning, on the C3 input
    gen = synth.gen_batch(range(200_000, 200_256), n_fr, synth.SceneSpec.dense())
    mixed = device_frames(gen, 0, 256, tile=4)
    half_a = device_frames(gen, 0, 256, tile=2)                 # scenes 0..511 of the mixed context
    one = BatchedTracker(S, max_points=1024, max_tracks=16)
    one.load_pose_weights(W)
    one.set_scene_trackers(scenes=slice(S // 2, S), tr_max_tracks=10)
    a = BatchedTracker(S // 2, max_points=1024, max_tracks=16)
    b = BatchedTracker(S // 2, max_points=1024, max_tracks=16, config=default_config(tr_max_tracks=10))
    for x in (a, b):
        x.load_pose_weights(W)
    t_one, t_two = [], []
    for f in range(n_fr):
        t0 = time.perf_counter()
        step(one, mixed[f])
        one.sync()
        t1 = time.perf_counter()
        step(a, half_a[f])
        step(b, half_a[f])
        a.sync()
        b.sync()
        t2 = time.perf_counter()
        if f >= args.warmup:
            t_one.append(t1 - t0)
            t_two.append(t2 - t1)
    _, nt = one.tracks()
    print("1024 dense scenes (C3 input), max_points 1024, max_tracks 16, half tr_max_tracks = 4 and half = 10, "
          "serial steps with pose; %.2f tracks per scene at the end" % nt.mean())
    print("  one context, mixed tracker table: %.3f ms per frame (median of %d)" % (1e3 * np.median(t_one), len(t_one)))
    print("  two contexts of 512, back to back: %.3f ms per frame (median of %d)" % (1e3 * np.median(t_two), len(t_two)))


if __name__ == "__main__":
    main()
