"""Cost of per-scene export / import (mmw_export_scenes, mmw_import_scenes) at the C2 shape (1024 scenes, 256 points per
frame, 8 tracks, 3-D pose net), after 30 frames so that the scenes hold live tracks.

Prints, with the GPU's name and power limit read in the same run:
  - the wall time of export and of import (host clock around each synchronous call) for n = 1, 16, 256 and 1024 scenes,
    with a pageable and with a pinned blob, median of --reps calls;
  - mmw_state_dump / mmw_state_restore of the whole context, for comparison;
  - the serial step time (CUDA events on the library's stream, L2 flushed before every timed step) of the blocks of
    steps just before and just after a move of 512 scenes between two contexts.
Run from the repository root: python profiles/scene_move.py
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
from mmwave_msc_b200.batched import BatchedTracker  # noqa: E402
from mmwave_msc_b200.sharding import move_scenes  # noqa: E402


def device_frames(S, n):
    out = []
    for b in synth.gen_batch(range(S), n):
        out.append((torch.from_numpy(b.points).cuda(), torch.from_numpy(b.offsets).cuda(), torch.from_numpy(b.dt).cuda()))
    return out


def wall(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=1024)
    ap.add_argument("--frames", type=int, default=30, help="frames stepped before the timings")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=30, help="timed steps before and after the move")
    args = ap.parse_args()
    S, R = args.scenes, args.reps
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    W = pw.make_pose_weights(pw.VARIANT_3D)
    a, b = (BatchedTracker(S, max_points=256, max_tracks=8) for _ in range(2))
    for bt in (a, b):
        bt.load_pose_weights(W)
    dev = device_frames(S, args.frames + 2 * args.steps)
    f = 0

    def step(bt):
        p, o, d = dev[f]
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True)

    for f in range(args.frames):
        step(a)
        step(b)
    a.sync()
    b.sync()
    n_tracks = a.summary()[0]
    print("GPU: %s" % gpu)
    print("C2 shape: %d scenes x (256 points, 8 tracks), 3-D pose net, after %d frames: %d live tracks; record %d bytes"
          % (S, args.frames, int(n_tracks.sum()), a.scene_state_size(1) - 64 - 16))
    print("wall time of one synchronous call, median of %d (host clock)" % R)
    print("%6s %12s %9s %11s %11s %11s %11s" % ("n", "blob bytes", "", "export ms", "GB/s", "import ms", "GB/s"))
    for n in (1, 16, 256, 1024):
        n = min(n, S)
        idx = np.arange(n, dtype=np.int32) * (S // n)
        size = a.scene_state_size(n)
        for kind in ("pageable", "pinned"):
            buf = np.empty(size, np.uint8) if kind == "pageable" else torch.empty(size, dtype=torch.uint8).pin_memory().numpy()
            a.export_scenes(idx, out=buf)                               # warm-up (grows the move buffer)
            b.import_scenes(buf, idx)
            te = wall(lambda: a.export_scenes(idx, out=buf), R)
            ti = wall(lambda: b.import_scenes(buf, idx), R)
            print("%6d %12d %9s %11.3f %11.2f %11.3f %11.2f" % (n, size, kind, te, size / te / 1e6, ti, size / ti / 1e6))
    blob = a.state_dump()
    td = wall(lambda: a.state_dump(), R)
    tr = wall(lambda: b.state_restore(blob), R)
    print("whole context (pageable): mmw_state_dump %.3f ms, mmw_state_restore %.3f ms, %d bytes" % (td, tr, blob.size))

    # serial step time of the blocks before and after a move of 512 scenes from a to b
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    stream = torch.cuda.ExternalStream(a.stream)

    def timed_block(f0):
        nonlocal f
        ev = []
        for k in range(args.steps):
            f = f0 + k
            with torch.cuda.stream(stream):
                flush.fill_(k & 0xff)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
            step(a)
            e1.record(stream)
            ev.append((e0, e1))
        a.sync()
        return np.array([x.elapsed_time(y) for x, y in ev])

    before = timed_block(args.frames)
    half = np.arange(0, S, 2, dtype=np.int32)
    t0 = time.perf_counter()
    move_scenes(a, half, b, half, reset_source=False)
    tm = 1e3 * (time.perf_counter() - t0)
    after = timed_block(args.frames + args.steps)
    print("move_scenes of %d scenes (export + import, pageable blob): %.3f ms" % (half.size, tm))
    print("serial step of the source context, %d steps each: before the move %.4f ms (median %.4f), after %.4f ms "
          "(median %.4f)" % (args.steps, before.mean(), np.median(before), after.mean(), np.median(after)))


if __name__ == "__main__":
    main()
