"""Packets to tracker at the C2 shape (1024 scenes, ~200 points per frame, 3-D pose net): three ways of running the
same frames, each in its own context, in serial and in throughput mode (MMW_STEP_PIPELINE), alternated in blocks of
--block steps in one run:
  packets      mmw_step_packets on the framed UART packets (pinned)
  decode+step  mmw_decode_tlv on the same packets (synchronous, rows back to the host), then mmw_step on those rows
  int16        mmw_step on int16 rows (x, y, z, dopplerIdx, peakVal; pinned), what a caller that decodes on the host sends
Scenes are synth.gen_scene frames encoded with oracle.tlv_oracle.encode_packet (one radar profile: 32 Doppler bins,
0.0626 m/s, Q9).  ms per step = host wall clock over a block, ending in a synchronise (decode+step blocks the host on
every call); L2 is not flushed.  Also prints the per-kernel time of the packet decode (MMW_K_PACKETS) and of step_kernel,
the GPU's name and power limit, and whether the three contexts end with the same tracks.
Run from the repository root: python profiles/packets_e2e.py
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from mmwave_msc_b200 import _lib, pose_weights as pw, synth  # noqa: E402
from mmwave_msc_b200.batched import BatchedTracker, concat_packets, default_config  # noqa: E402
from oracle import tlv_oracle as tlv  # noqa: E402

BINS, RES, Q = 32, 0.0626, 9


def pinned(a):
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t, t.numpy()


def int16_rows(blob, off):
    """The rows a host-side decoder would send with MMW_STEP_INPUT_I16 (ReadIWR14xx.read's words, Doppler corrected)."""
    rows = []
    for s in range(len(off) - 1):
        p = bytes(blob[off[s]:off[s + 1]])
        ok, _, _ = tlv.decode_packet(p, BINS, RES)
        if not ok:
            rows.append(np.zeros((0, 5), np.int16))
            continue
        n = int.from_bytes(p[44:46], "little")
        w = np.frombuffer(p, "<i2", count=6 * n, offset=48).reshape(n, 6).astype(np.int16)
        d = w[:, 1].astype(np.int32)
        d = np.where(d > BINS / 2 - 1, (d - 65535).astype(np.int16), d)
        rows.append(np.stack([w[:, 3], w[:, 4], w[:, 5], d.astype(np.int16), w[:, 2]], axis=1))
    r_off = np.zeros(len(rows) + 1, np.int32)
    r_off[1:] = np.cumsum([len(r) for r in rows])
    return np.concatenate(rows, axis=0), r_off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=1024)
    ap.add_argument("--frames", type=int, default=40, help="distinct frames (cycled)")
    ap.add_argument("--steps", type=int, default=120, help="timed steps per arm and mode")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--block", type=int, default=10, help="steps per arm between switches")
    args = ap.parse_args()
    S, NF = args.scenes, args.frames
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    scenes = [synth.gen_scene(s, NF, synth.SceneSpec(doppler_res=RES)) for s in range(S)]
    frames = []
    for f in range(NF):
        blob, off = concat_packets([tlv.encode_packet(f + 1, sc.frames[f], Q, RES) for sc in scenes])
        i16, i16_off = int16_rows(blob, off)
        dt = np.array([sc.dts()[f] for sc in scenes])
        frames.append({"blob": pinned(blob), "off": pinned(off), "i16": pinned(i16), "i16_off": pinned(i16_off),
                       "dt": pinned(dt)})
    n_pts = np.mean([fr["i16_off"][1][-1] for fr in frames])
    weights = pw.make_pose_weights(pw.VARIANT_3D)
    lib = _lib.load()
    arms = {}
    for name in ("packets", "decode+step", "int16"):
        bt = BatchedTracker(S, max_points=256, max_tracks=8, config=default_config(doppler_res=RES))
        bt.load_pose_weights(weights)
        bt.set_scene_sensors(num_doppler_bins=BINS)
        arms[name] = {"bt": bt, "f": 0, "ms": {"serial": [], "throughput": []}}
    cap = S * 256
    dec = {"pts": np.zeros((cap, 5), np.float32), "poff": np.zeros(S + 1, np.int32), "fr": np.zeros(S, np.int32),
           "ok": np.zeros(S, np.int32)}

    def step(name, pipe):
        a = arms[name]
        fr = frames[a["f"] % NF]
        a["f"] += 1
        h = a["bt"]._h
        flags = _lib.STEP_POSE | (_lib.STEP_PIPELINE if pipe else 0)
        if name == "packets":
            rc = lib.mmw_step_packets(h, _lib.ptr(fr["blob"][1]), _lib.ptr(fr["off"][1]), _lib.ptr(fr["dt"][1]), flags,
                                      None, None)
        elif name == "decode+step":
            rc = lib.mmw_decode_tlv(h, _lib.ptr(fr["blob"][1]), _lib.ptr(fr["off"][1]), S, float(BINS), RES,
                                    _lib.ptr(dec["pts"]), cap, _lib.ptr(dec["poff"]), _lib.ptr(dec["fr"]),
                                    _lib.ptr(dec["ok"]))
            _lib.check(rc)
            rc = lib.mmw_step(h, _lib.ptr(dec["pts"]), _lib.ptr(dec["poff"]), _lib.ptr(fr["dt"][1]), flags)
        else:
            rc = lib.mmw_step(h, _lib.ptr(fr["i16"][1]), _lib.ptr(fr["i16_off"][1]), _lib.ptr(fr["dt"][1]),
                              flags | _lib.STEP_INPUT_I16)
        _lib.check(rc)

    for mode in ("serial", "throughput"):
        for name in arms:
            for _ in range(args.warmup):
                step(name, mode == "throughput")
            arms[name]["bt"].sync()
    for b0 in range(0, args.steps, args.block):
        nb = min(args.block, args.steps - b0)
        for mode in ("serial", "throughput"):
            for name, a in arms.items():
                a["bt"].sync()
                t0 = time.perf_counter()
                for _ in range(nb):
                    step(name, mode == "throughput")
                a["bt"].sync()
                a["ms"][mode].append((time.perf_counter() - t0) * 1e3 / nb)
    tracks = {name: a["bt"].tracks()[0].tobytes() for name, a in arms.items()}
    print("GPU: %s" % gpu)
    print("C2 shape: %d scenes, %.1f points per scene-frame, pose on, %d timed steps per arm and mode in blocks of %d"
          % (S, n_pts / S, args.steps, args.block))
    print("same tracks in all three contexts: %s" % (len(set(tracks.values())) == 1))
    for mode in ("serial", "throughput"):
        for name, a in arms.items():
            ms = np.array(a["ms"][mode])
            print("%-10s  %-11s  %.4f ms/step  (median of blocks %.4f, min %.4f, max %.4f)"
                  % (mode, name, ms.mean(), np.median(ms), ms.min(), ms.max()))
    for name in ("packets", "int16"):
        kern = arms[name]["bt"].profile_kernels(lambda i, name=name: step(name, False), 20)
        print("kernels (serial, %s): %s" % (name, "  ".join("%s %.4f ms" % kv for kv in kern.items())))


if __name__ == "__main__":
    main()
