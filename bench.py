#!/usr/bin/env python
"""Benchmark of the per-frame radar perception path (cluster + track + pose) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one radar frame for every resident scene: Utils.normalize_data -> TrackBuffer.track ->
TrackBuffer.estimate_posture of the reference (offline_main.py:45-60), S scenes at once per GPU.
Workload = BASELINE config C2 per GPU (1024 concurrent synthetic IWR1443-shaped scenes, ~200 pts/frame, up to 4
tracks each, reference default constants => the 3-frame 3-D pose net); with N GPUs the scenes are sharded
1024 per GPU (N=8 is BASELINE config C5, 8192 scenes), no inter-GPU traffic in the hot loop, one NCCL
all-gather of the packed results at the end.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCENES_PER_GPU = 1024
PRIME_FRAMES = 12          # untimed frames before warm-up so that tracks exist (start-up DBSCAN is not steady state)
METRIC = "radar frames/sec (cluster+track+pose)"
UNIT = "scene-frames/s"
WORKLOAD = ("C2: %d concurrent synthetic IWR1443 scenes per GPU, ~200 pts/frame (U{160..240}), 1-4 people, "
            "12 Hz cfg, reference default constants (FB_FRAMES_BATCH=2 -> 3x8x8x5 pose net)" % SCENES_PER_GPU)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "src": "measured (MEASURED_PEAKS.json; bf16 = sustained, kernel timed inside a long step)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "src": "fallback (B200_PROFILING.md)"}


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons DURING the timed regions (B200_PROFILING.md recipe).
    Sampled through NVML in a thread of this process every 5 ms: the same counters `nvidia-smi --query-gpu=clocks.sm,
    clocks.max.sm,power.draw,clocks_event_reasons.*` prints, without a second process polling the driver -- the
    nvidia-smi loop stalled the launch path for milliseconds at a time, which is a third of a 5 ms timed window.
    Falls back to that loop when NVML cannot be loaded."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows, self.samples = [], []
        self.proc = None
        self.nvml = None
        self.stop_flag = False

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except Exception:
                pass
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self._physical_index()), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1e3
                rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.stop_flag = True
            self.th.join(timeout=1)
            n = self.nvml
            bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            reasons = sorted(k for k, b in bits.items() if any(s[2] & b for s in self.samples))
            sm = [s[0] for s in self.samples]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.sm_max,
                    "power_w_max": max((s[1] for s in self.samples), default=None), "samples": len(sm),
                    "reasons": reasons, "source": "NVML (in-process, every 5 ms)"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi -lms 20"}


# --------------------------------------------------------------------------------------------------
def algorithmic_bytes(cnt: np.ndarray, nfr: int) -> float:
    """SURVEY.md section 8(d) per scene-frame formula summed from the device counters:
    20 N + 4 M + 32 U + 32 Bf[dbscan ran] + sum_tracks (2*624 + 20 min(A_j,64) + nfr*64*20 + 228) + 8."""
    frames, N, M, U, Bf, T, rows, pose = (float(x) for x in cnt)
    return 20 * N + 4 * M + 32 * U + 32 * Bf + T * (2 * 624 + nfr * 64 * 20 + 228) + 20 * rows + 8 * frames


def cpu_port_run(scene_ids, n_frames, with_pose=True):
    """The oracle port (numpy restatement of the reference path) on the given scenes; returns scene-frames, seconds."""
    from mmwave_msc_b200 import pose_weights as pw, synth
    from oracle import mmw_oracle as mo
    try:
        import torch
        torch.set_num_threads(1)
    except Exception:
        pass
    W = pw.make_pose_weights(pw.VARIANT_3D) if with_pose else None
    scenes = [synth.gen_scene(s, n_frames) for s in scene_ids]
    t0 = time.perf_counter()
    n = 0
    for sc in scenes:
        so = mo.SceneOracle(pose_weights=W, pose_dtype=np.float32)
        for fr, dt in zip(sc.frames, sc.dts()):
            so.step(fr, dt)
            n += 1
    return n, time.perf_counter() - t0


def _cpu_worker(args):
    os.environ["OMP_NUM_THREADS"] = "1"
    return cpu_port_run(*args)


def reference_run(scene_ids, n_frames):
    """The reference ITSELF (unmodified Utils.normalize_data / TrackBuffer.track / estimate_posture from
    oracle/_ref/src -- staged by oracle/make_ref.py -- or /root/reference/src), driven by the loop body of
    offline_main.py:45-60: sklearn DBSCAN as shipped (BallTree), default argsort.  filterpy is the restatement of
    oracle/filterpy_shim, the Keras model a torch-CPU fp32 module behind .predict (neither library is installed).
    Returns scene-frames, seconds."""
    from mmwave_msc_b200 import pose_weights as pw, synth
    from oracle import mmw_oracle as mo, ref_harness as rh
    try:
        import torch
        torch.set_num_threads(1)
    except Exception:
        pass
    const, utils, tracking = rh.load_reference()
    W = pw.make_pose_weights(pw.VARIANT_3D)

    class Model:
        def predict(self, x):
            return mo.pose_forward(W, np.asarray(x, np.float32), np.float32)

    scenes = [synth.gen_scene(s, n_frames) for s in scene_ids]
    dets = [[rh.detobj_from_raw(fr) for fr in sc.frames] for sc in scenes]
    model = Model()
    devnull = open(os.devnull, "w")
    out, sys.stdout = sys.stdout, devnull          # the reference prints on malformed points (Utils.py:398)
    try:
        t0 = time.perf_counter()
        n = 0
        for sc, dd in zip(scenes, dets):
            tb, batch = tracking.TrackBuffer(), tracking.BatchedData()
            for det, dt in zip(dd, sc.dts()):
                tb.dt = float(dt)
                eff = utils.normalize_data(det)
                if eff.shape[0] != 0:
                    tb.track(eff, batch)
                    tb.estimate_posture(model)
                n += 1
        sec = time.perf_counter() - t0
    finally:
        sys.stdout = out
    return n, sec


def _ref_worker(args):
    os.environ["OMP_NUM_THREADS"] = "1"
    return reference_run(*args)


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on all host cores, independent scenes per
    process (the reference is single-threaded).  Uses the staged unmodified reference (kind "reference"); without it
    the oracle port (kind "port", ~10x faster than the real thing)."""
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import make_ref
    real = bool(make_ref.staged_dir())
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    frames = 30
    per_proc = 1 if real else 2
    vals = []
    for step in range(args.warmup + args.steps):
        jobs = [([10_000 + step * 1000 + p * per_proc + i for i in range(per_proc)], frames) for p in range(procs)]
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_ref_worker if real else _cpu_worker_pose, jobs)
        wall = max(r[1] for r in res)
        if step >= args.warmup:
            vals.append(sum(r[0] for r in res) / wall)
    v = float(np.mean(vals)) if vals else 0.0
    impl = ("the unmodified reference (Utils.normalize_data, TrackBuffer.track, estimate_posture; offline_main.py "
            "loop body) with the filterpy restatement and a torch-CPU fp32 pose net behind .predict"
            if real else "oracle port (numpy float64 + torch-CPU fp32 pose net)")
    sample = "%d processes x %d scene(s) x %d frames per step (C2-shaped scenes), %s" % (procs, per_proc, frames, impl)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * procs * per_proc * frames / v if v else None,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": "reference" if real else "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def _cpu_worker_pose(args):
    os.environ["OMP_NUM_THREADS"] = "1"
    return cpu_port_run(args[0], args[1], True)


# --------------------------------------------------------------------------------------------------
def pin_to_gpu_numa_node(local):
    """Best effort: run this rank (and place its pinned buffers, first touch) on the cores of the NUMA node its GPU
    hangs off.  Returns a description for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return {"numa_node": None, "why": "the platform reports no NUMA node for %s" % bus}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "why": "no allowed core on that node"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cores": len(cpus), "gpu": bus}
    except Exception as e:                      # never fatal: it is an optimisation
        return {"numa_node": None, "why": "%s: %s" % (type(e).__name__, e)}


DOPPLER_RES = 0.0626       # Doppler bin of the 12 Hz profile the synthetic generator quantises to (synth.py)


def lattice_rows(points):
    """The generator's fp32 rows as the sensor's lattice: (fp32 rows with the Doppler column as the index, int16 rows
    x, y, z in Q9, dopplerIdx, peakVal).  The context multiplies the index by mmw_config::doppler_res in float64."""
    p = points.astype(np.float64)
    q = np.stack([np.rint(p[:, 0] * 512), np.rint(p[:, 1] * 512), np.rint(p[:, 2] * 512), np.rint(p[:, 3] / DOPPLER_RES),
                  np.rint(p[:, 4])], axis=1)
    f32 = np.stack([q[:, 0] / 512, q[:, 1] / 512, q[:, 2] / 512, q[:, 3], q[:, 4]], axis=1).astype(np.float32)
    return np.ascontiguousarray(f32), np.ascontiguousarray(q.astype(np.int16))


def _tile_batches(batches, reps):
    """The same scenes `reps` times side by side (scene s + k * S is scene s again): a throughput workload of
    reps * S scenes from S generated ones."""
    out = []
    for b in batches:
        n = b.points.shape[0]
        pts = np.tile(b.points, (reps, 1))
        off = np.concatenate([b.offsets[:-1] + k * n for k in range(reps)] + [np.array([reps * n], np.int32)])
        out.append((pts, off.astype(np.int32), np.tile(b.dt, reps)))
    return out


def _timed_device_steps(bt, host_batches, prime, warm, K, flush, local):
    """Device-resident inputs, L2 flushed before every timed step, CUDA events on the library's stream."""
    import torch
    stream = torch.cuda.ExternalStream(bt.stream, device=local)
    ms = []
    for f, (pts, off, dt) in enumerate(host_batches[:prime + warm + K]):
        p, o, d = torch.from_numpy(pts).cuda(), torch.from_numpy(off).cuda(), torch.from_numpy(dt).cuda()
        timed = f >= prime + warm
        with torch.cuda.stream(stream):
            if timed:
                flush.fill_(f & 0xff)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
            bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True)
            if timed:
                e1.record(stream)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
        bt.sync()
    return np.array(ms)


def _timed_device_pipeline(bt, host_batches, warm, K, local):
    """Throughput mode (MMW_STEP_PIPELINE) on a context that has already been primed: device-resident inputs, K steps
    on frames never read before inside one pair of CUDA events (the second after the streams have joined)."""
    import torch
    from mmwave_msc_b200 import _lib
    stream = torch.cuda.ExternalStream(bt.stream, device=local)
    dev = [(torch.from_numpy(p).cuda(), torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda())
           for p, o, d in host_batches[:warm + K]]
    res = torch.empty(bt.S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    for p, o, d in dev[:warm]:
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=True)
    bt.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for p, o, d in dev[warm:]:
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=True)
    bt.pack_results(res.data_ptr())               # serial-mode call: the main stream waits for the pose stream first
    e1.record(stream)
    bt.sync()
    return e0.elapsed_time(e1) / K


def other_configs(batches, weights3d, flush, local):
    """The BASELINE.json configurations that are not the headline workload, on ONE GPU (same timing protocol):
    C3 dense 8.5 m (1000 points/frame, 10 targets, TR_MAX_TRACKS = 10), C4 pose regression alone (65 536 maps,
    2-D net), C5 all 8192 scenes on one GPU.  C1 (one scene) is `latency.p50_ms_single_scene_*`."""
    from mmwave_msc_b200 import _lib, pose_weights as pw, synth
    from mmwave_msc_b200.batched import BatchedTracker, default_config
    from oracle import mmw_oracle as mo
    PRIME, WARM, K = 12, 3, 8
    out = {}
    # C3
    gen = synth.gen_batch(range(200_000, 200_256), PRIME + 2 * (WARM + K), synth.SceneSpec.dense())
    tiled = _tile_batches(gen, 4)
    bt = BatchedTracker(1024, max_points=1024, max_tracks=16, device=local, config=default_config(tr_max_tracks=10))
    bt.load_pose_weights(weights3d)
    ms = _timed_device_steps(bt, tiled, PRIME, WARM, K, flush, local)
    _, nt = bt.tracks()
    tp = _timed_device_pipeline(bt, tiled[PRIME + WARM + K:], WARM, K, local)
    out["C3"] = {"what": "dense 8.5 m config: 1024 scenes (256 generated x 4), 1000 points/frame, 10 targets, "
                         "TR_MAX_TRACKS = 10, full path incl. pose", "scenes": 1024,
                 "points_per_scene_frame": float(np.mean([t[0].shape[0] for t in tiled]) / 1024),
                 "tracks_per_scene": float(nt.mean()), "ms_per_step": float(ms.mean()),
                 "scene_frames_per_s": float(1024 / (ms.mean() / 1e3)),
                 "throughput_mode": {"ms_per_step": tp, "scene_frames_per_s": float(1024 / (tp / 1e3))}}
    bt.close()
    # C5 on one GPU: the headline run's own scenes, eight times side by side
    tiled = _tile_batches(batches[:PRIME + 2 * (WARM + K)], 8)
    bt = BatchedTracker(8192, max_points=256, max_tracks=8, device=local,
                        config=default_config(doppler_res=DOPPLER_RES, xyz_q_format=9))
    bt.load_pose_weights(weights3d)
    ms = _timed_device_steps(bt, tiled, PRIME, WARM, K, flush, local)
    tp = _timed_device_pipeline(bt, tiled[PRIME + WARM + K:], WARM, K, local)
    out["C5_one_gpu"] = {"what": "8192 scenes on ONE GPU (the 1024 generated scenes x 8), full path incl. pose",
                         "scenes": 8192, "ms_per_step": float(ms.mean()),
                         "scene_frames_per_s": float(8192 / (ms.mean() / 1e3)),
                         "throughput_mode": {"ms_per_step": tp, "scene_frames_per_s": float(8192 / (tp / 1e3))}}
    # C4 on the same context size: 65 536 feature maps through the 2-D net
    bt.close()
    N = 65536
    rng = np.random.default_rng(4)
    k = rng.integers(20, 65, size=N)
    rows = np.zeros((N, 64, 5), np.float32)
    rows[:, :, :3] = rng.normal([0, 0, 1.0], [0.15, 0.15, 0.4], size=(N, 64, 3))
    rows[:, :, 3] = rng.normal(0, 0.3, size=(N, 64))
    rows[:, :, 4] = (np.floor(rng.gamma(0.5, 54.0, size=(N, 64))) + 1 - 27.0187) / 70.351
    rows[np.arange(64)[None, :] >= k[:, None]] = 0.0                    # zero pads after the real rows
    order = np.argsort(rows[:, :, 0], axis=1, kind="stable")
    feats = np.take_along_axis(rows, order[:, :, None], axis=1).reshape(N, 8, 8, 5)
    W2 = pw.make_pose_weights(pw.VARIANT_2D)
    bt = BatchedTracker(8192, max_tracks=8, device=local, config=default_config(frames_batch=0))
    bt.load_pose_weights(W2, pw.VARIANT_2D)
    got = bt.pose(feats)
    err = float(np.abs(got[:256] - mo.pose_forward(W2, feats[:256], np.float64)).max())
    _lib.check(bt.lib.mmw_profile(bt._h, 1))
    for _ in range(5):
        bt.pose(feats)
    kms = np.zeros(8); calls = np.zeros(8, np.uint64)
    _lib.check(bt.lib.mmw_get_kernel_ms(bt._h, _lib.ptr(kms), _lib.ptr(calls)))
    _lib.check(bt.lib.mmw_profile(bt._h, 0))
    per = {n: float(kms[i] / calls[i]) for i, n in enumerate(_lib.KERNEL_NAMES) if calls[i]}
    total = sum(per.values())
    out["C4"] = {"what": "MARS-style pose regression alone: 65 536 8x8x5 maps -> 57 (define_CNN, tcgen05 path), device "
                         "time of the pose kernels (CUDA events around every launch)", "rows": N, "kernel_ms": per,
                 "pose_ms": total, "maps_per_s": N / (total / 1e3),
                 "algorithmic_tflops": 2837504.0 * N / (total / 1e3) / 1e12,
                 "max_joint_err_m_vs_fp64_oracle_256_rows": err}
    bt.close()
    return out


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(bt, offsets, out_dir):
    """Writes what a caller of the timed path holds after its last step as out_dir/<name>.npy: every field of the track
    records (mmw_get_tracks) and the track counts, the packed result records (mmw_pack_results), the per-scene status
    flags and the association of every input point of the frame (with the frame's scene offsets).  Integers are stored
    as float64, which holds them exactly.  Above DUMP_BYTES_MAX in all, a fixed seeded sample of the scenes is written;
    scene_index lists the scenes written."""
    import torch
    from mmwave_msc_b200 import _lib
    tr, nt = bt.tracks()
    res = torch.empty(bt.S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32, device="cuda")
    bt.pack_results(res.data_ptr())
    bt.sync()
    out = {"n_tracks": nt, "status": bt.status(), "results": res.cpu().numpy().reshape(bt.S, bt.tcap, -1)}
    out.update(("track_" + k, tr[k]) for k in tr.dtype.names if not k.startswith("reserved"))
    out = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in out.items()}
    assoc = bt.point_assoc().astype(np.float64)
    per_scene = sum(v.nbytes for v in out.values()) // bt.S + 8 * bt.ncap + 24
    budget = DUMP_BYTES_MAX - (1 << 20)                  # room for the .npy headers
    scenes = np.arange(bt.S)
    if per_scene * bt.S > budget:
        scenes = np.sort(np.random.default_rng(0).choice(bt.S, budget // per_scene, replace=False))
    out = {k: v[scenes] for k, v in out.items()}
    out["point_assoc"] = np.concatenate([assoc[offsets[s]:offsets[s + 1]] for s in scenes])
    out["point_offsets"] = np.concatenate([[0], np.cumsum(offsets[scenes + 1] - offsets[scenes])]).astype(np.float64)
    out["scene_index"] = scenes.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(v))


def replay_check(world, S, n_frames_done, weights, gathered, per_scene, local, pose_calls):
    """SURVEY 8(e): a scene's results do not depend on which GPU ran it.  Rank 0 re-runs the first scenes of rank 1's
    shard from frame 0 through the same sequence of calls in a context of its own and compares the records with
    the ones rank 1 contributed to the gather -- bitwise."""
    from mmwave_msc_b200 import _lib, synth
    from mmwave_msc_b200.batched import BatchedTracker
    import torch
    n_check = min(32, S)
    ids = list(range(S, S + n_check))                     # global scene ids of rank 1's first scenes
    from mmwave_msc_b200.batched import default_config
    batches = synth.gen_batch(ids, n_frames_done)
    bt = BatchedTracker(n_check, max_points=256, max_tracks=8, device=local,
                        config=default_config(doppler_res=DOPPLER_RES, xyz_q_format=9))
    bt.load_pose_weights(weights)
    for f, b in enumerate(batches):
        bt.step(lattice_rows(b.points)[1], b.offsets, b.dt, pose=pose_calls[f])        # int16 rows, serial mode
    out = torch.empty(n_check * per_scene, dtype=torch.float32, device="cuda")
    bt.pack_results(out.data_ptr())
    bt.sync()
    mine = out.cpu().numpy().view(np.uint32)
    theirs = gathered[S * per_scene:(S + n_check) * per_scene].cpu().numpy().view(np.uint32)
    bt.close()
    return {"scenes_compared": n_check, "of_rank": 1, "frames": n_frames_done,
            "bitwise_identical": bool(np.array_equal(mine, theirs)),
            "mismatching_words": int((mine != theirs).sum())}


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--scenes", type=int, default=SCENES_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dense-path", default="tc", choices=["tc", "simt"])
    ap.add_argument("--no-l2-flush", action="store_true", help="diagnostic only: keep L2 warm between timed steps")
    ap.add_argument("--e2e-full-records", action="store_true",
                    help="end-to-end pass downloads all S * max_tracks records per frame instead of the live ones")
    ap.add_argument("--e2e-reps", type=int, default=5, help="end-to-end windows of K steps (the median is reported)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed (rank 0's scenes) to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path, not of --impl reference")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner with
    # printf whatever NCCL_DEBUG_FILE says): from here on file descriptor 1 IS stderr, and the JSON line goes to the
    # saved original at the end.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    _print = print

    def emit(*a, **k):
        _print(*a, file=real_stdout, **k)
        real_stdout.flush()

    globals()["print"] = emit
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    # the contract is ONE JSON line on stdout: NCCL's own debug output (whatever level the caller asked for) goes
    # to stderr, not to stdout
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    from mmwave_msc_b200 import _lib, pose_weights as pw, sharding, synth
    from mmwave_msc_b200.batched import BatchedTracker

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa = pin_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    S = args.scenes
    W_, K = args.warmup, args.steps
    LAT_FRAMES = 12
    E2E_REPS = max(1, args.e2e_reps)   # the end-to-end window of K steps is ~5 ms: measured this many times, median reported
    n_frames = PRIME_FRAMES + 2 * (W_ + K) + (W_ + E2E_REPS * K) + K + LAT_FRAMES   # device-timed, throughput-mode, e2e, latency, per-kernel profile
    ids = sharding.shard_scene_ids(world * S, world, rank)      # contiguous block of scenes per GPU
    batches = synth.gen_batch(ids, n_frames)
    # the sensor's lattice: fp32 rows for the device-resident passes, int16 rows (10 bytes per point) for the end-to-end
    # pass; the Doppler column is the index, the context multiplies by the resolution in float64
    rows16 = []
    for b in batches:
        b.points, r16 = lattice_rows(b.points)
        rows16.append(r16)

    from mmwave_msc_b200.batched import default_config
    bt = BatchedTracker(S, max_points=256, max_tracks=8, device=local,
                        config=default_config(doppler_res=DOPPLER_RES, xyz_q_format=9))
    weights = pw.make_pose_weights(pw.VARIANT_3D)
    bt.load_pose_weights(weights)
    bt.set_dense_path(args.dense_path == "tc")
    stream = torch.cuda.ExternalStream(bt.stream, device=local)

    # inputs resident in HBM for the device-timed pass; pinned host copies for the end-to-end pass
    dev = []
    for b in batches:
        dev.append((torch.from_numpy(b.points).cuda(), torch.from_numpy(b.offsets).cuda(), torch.from_numpy(b.dt).cuda()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    torch.cuda.synchronize()

    def step_dev(f, pose=True):
        p, o, d = dev[f]
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=pose)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    f = 0
    for _ in range(PRIME_FRAMES):
        step_dev(f); f += 1
    for _ in range(W_):
        step_dev(f); f += 1
    bt.sync()
    bt.counters(reset=True)
    launches0 = bt.launch_count()

    # ---- device-timed pass: K steps, inputs resident in HBM, L2 flushed between steps ----------------------
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    # The steps are queued in chunks of five behind a ~10 ms spin kernel, so that the device runs them back to back
    # whatever the host is doing (with several ranks on one box a descheduled host thread otherwise shows up INSIDE a
    # step, between two of its kernels); the library's host-side hints (work-list length, pose-row count) are refreshed
    # between the chunks as they would be in a live loop.
    CHUNK = 5
    for c0 in range(0, K, CHUNK):
        with torch.cuda.stream(stream):
            torch.cuda._sleep(20_000_000)
        for k in range(c0, min(K, c0 + CHUNK)):
            with torch.cuda.stream(stream):
                if not args.no_l2_flush:
                    flush.fill_(k & 0xff)        # evict L2 between timed iterations (not inside the timed interval)
                ev[k][0].record(stream)
            step_dev(f); f += 1
            ev[k][1].record(stream)
        bt.sync()
    barrier()
    step_ms = np.array([a.elapsed_time(b) for a, b in ev])
    total_ms = float(step_ms.sum())
    launches = bt.launch_count() - launches0
    cnt = bt.counters(reset=True)
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * S * K / (total_ms_max / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(bt, batches[f - 1].offsets, args.dump_outputs)

    # ---- per-kernel durations (CUDA events on the library's stream around every launch), on the K frames that follow
    # the device-timed ones: the track count rises slowly over a sequence, and the roofline figures must describe the
    # same regime as `value`
    kern = bt.profile_kernels(lambda i: step_dev(f + i), K)
    f += K
    bt.sync()
    bt.counters(reset=True)

    # ---- throughput mode (MMW_STEP_PIPELINE): the pose network of frame k on a second stream under the tracker of
    # frame k + 1 (results bit-identical to the serial mode); K steps back to back, device-resident inputs, one pair of
    # CUDA events around all of them (the second after the main stream has joined the pose stream), max over ranks.
    # No explicit L2 flush here -- a fill on either stream would serialise them: every step reads a frame that has never
    # been read before from its own buffer and streams ~150 MB of state, activations and weights through the 126 MB L2.
    # Reported next to the headline `value`, which stays the serial, flushed, per-step protocol.
    res_dev0 = torch.empty(S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32, device="cuda")
    for _ in range(W_):
        p, o, d = dev[f]
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=True); f += 1
    barrier(); bt.sync()
    t_ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    barrier()
    t_ev[0].record(stream)
    for k in range(K):
        p, o, d = dev[f]
        bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=True); f += 1
    bt.pack_results(res_dev0.data_ptr())          # serial-mode call: the main stream waits for the pose stream first
    t_ev[1].record(stream)
    barrier(); bt.sync()
    bt.counters(reset=True)
    tp_ms = torch.tensor([t_ev[0].elapsed_time(t_ev[1])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tp_ms, op=dist.ReduceOp.MAX)
    tp_ms = float(tp_ms.item())

    # ---- end-to-end pass through the public API: pinned host inputs, result read back every step ----------
    res_dev = torch.empty(S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32, device="cuda")
    per_frame = S * bt.tcap * _lib.RESULT_FLOATS

    # The public API for a replay of many scenes is mmw_run_frames (BatchedTracker.run_frames): the loop of
    # offline_main.py:40-62 in C over pinned host buffers -- int16 sensor rows up, packed result records down, every
    # frame's bytes crossing PCIe inside the timed region; uploads on one side stream into double-buffered staging, the
    # tracker on the main stream, the pose network on a second one (throughput mode), downloads on a third, so
    # upload(k+1) / tracker(k+1) / pose(k) / download(k-1) overlap.
    # Host buffers of all windows come from ONE pinned allocation per array, with a guard region behind the last
    # window: frames whose buffers lie in the most recently allocated pinned block ran 30 % slower in every run
    # (profiles/r02_e2e_last_window.txt: a property of the host allocation, gone as soon as anything is allocated
    # behind it).
    lo_all, hi_all = f, f + W_ + E2E_REPS * K
    n_all = hi_all - lo_all
    guard = 4
    rows_all = torch.from_numpy(np.concatenate(rows16[lo_all:hi_all] + [rows16[hi_all - 1]] * guard)).pin_memory().numpy()
    fro_all = np.cumsum([0] + [len(r) for r in rows16[lo_all:hi_all]]).astype(np.int64)
    offs_all = torch.from_numpy(np.stack([b.offsets for b in batches[lo_all:hi_all]] + [batches[hi_all - 1].offsets] * guard)).pin_memory().numpy()
    dts_all = torch.from_numpy(np.stack([b.dt for b in batches[lo_all:hi_all]] + [batches[hi_all - 1].dt] * guard)).pin_memory().numpy()
    res_all = torch.empty((n_all + guard, per_frame), dtype=torch.float32).pin_memory().numpy()
    cnt_all = torch.zeros(n_all + guard, dtype=torch.int32).pin_memory().numpy()

    def pinned_block(lo, hi):
        a, b = lo - lo_all, hi - lo_all
        return (rows_all[fro_all[a]:fro_all[b]], (fro_all[a:b + 1] - fro_all[a]).astype(np.int64), offs_all[a:b], dts_all[a:b],
                res_all[a:b], cnt_all[a:b])

    def run_block(blk):                # live records only (mmw_run_frames_compact) unless --e2e-full-records
        if args.e2e_full_records:
            bt.run_frames(*blk[:5])
        else:
            bt.run_frames(*blk[:5], n_records=blk[5])

    warm_blk = pinned_block(f, f + W_)
    time_blks = [pinned_block(f + W_ + r * K, f + W_ + (r + 1) * K) for r in range(E2E_REPS)]
    run_block(warm_blk)
    e2e_reps = []
    for blk in time_blks:              # consecutive frames of the same sequences: every window is K new frames
        barrier()
        t0 = time.perf_counter()
        run_block(blk)
        barrier()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_reps.append(float(t.item()))
    time_blk = time_blks[-1]
    h2d = time_blk[0].nbytes + time_blk[2].nbytes + time_blk[3].nbytes
    res_np = [time_blk[4][0], time_blk[4][1]]
    d2h = int(per_frame * 4) if args.e2e_full_records else int(time_blk[5].mean() * _lib.RESULT_FLOATS * 4 + 4)
    clocks = sampler.stop()           # sampled across the device-timed passes and the end-to-end pass
    clocks["window"] = "device-timed passes + end-to-end pass (all under load)"
    f += W_ + E2E_REPS * K
    e2e_value = world * S * K / float(np.median(e2e_reps))

    # ---- per-frame latency, host enqueue -> results in host memory, NOT pipelined (SURVEY 8(d)) -------------
    lat = []
    for i in range(LAT_FRAMES):
        b = batches[f + i]
        hp = (torch.from_numpy(b.points).pin_memory().numpy(), torch.from_numpy(b.offsets).pin_memory().numpy(),
              torch.from_numpy(b.dt).pin_memory().numpy())
        bt.sync()
        t0 = time.perf_counter()
        bt.step(*hp, pose=True)
        bt.wait_results(bt.read_results_async(res_np[0]))
        lat.append((time.perf_counter() - t0) * 1e3)
    f += LAT_FRAMES
    latency = {"p50_ms_step_device": float(np.median(step_ms)),
               "p50_ms_host_enqueue_to_results": float(np.median(lat[2:])),
               "note": "one frame of all %d scenes of this GPU; the second figure includes the upload from pinned "
                       "memory, the kernels, the result pack and its download, nothing overlapped" % S}
    if rank == 0:
        # C1: a single scene, what one live 12 Hz sensor would see
        one = BatchedTracker(1, max_points=256, max_tracks=8, device=local)
        one.load_pose_weights(weights)
        ob = synth.gen_batch([10_000], 40)
        r1 = torch.empty(one.tcap * _lib.RESULT_FLOATS, dtype=torch.float32).pin_memory().numpy()
        l1 = []
        for b in ob:
            hp = (torch.from_numpy(b.points).pin_memory().numpy(), torch.from_numpy(b.offsets).pin_memory().numpy(),
                  torch.from_numpy(b.dt).pin_memory().numpy())
            one.sync()
            t0 = time.perf_counter()
            one.step(*hp, pose=True)
            one.wait_results(one.read_results_async(r1))
            l1.append((time.perf_counter() - t0) * 1e3)
        latency["p50_ms_single_scene_host_enqueue_to_results"] = float(np.median(l1[10:]))
        one.close()

    # ---- final result gather: the only collective of the path (NCCL all-gather over NVLink) ---------------
    bt.pack_results(res_dev.data_ptr())
    bt.sync()
    if world > 1:
        gathered = sharding.gather_results(res_dev, world * S, bt.tcap * _lib.RESULT_FLOATS)
        torch.cuda.synchronize()
        assert gathered.numel() == world * res_dev.numel()
        # own shard comes back unchanged; another rank's scenes re-run here give the same bits (SURVEY 8(e))
        assert torch.equal(gathered[rank * res_dev.numel():(rank + 1) * res_dev.numel()], res_dev)
        identity = (replay_check(world, S, n_frames, weights, gathered, bt.tcap * _lib.RESULT_FLOATS, local,
                                 [True] * n_frames) if rank == 0 else None)
        # the same gather through the C ABI (mmw_gather_nccl: one ncclAllGather on the library's stream)
        ng = sharding.NcclGather(bt)
        via_abi = ng.gather()
        bt.sync()
        same = bool(torch.equal(via_abi, gathered))
        ng.close()
        if identity is not None:
            identity["mmw_gather_nccl_equals_torch_all_gather"] = same
        assert same, "mmw_gather_nccl and torch.distributed all_gather disagree"

    if rank == 0:
        pk = peaks()
        nfr = 3
        alg = algorithmic_bytes(cnt, nfr)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_,
            "ms_per_step": total_ms_max / K, "p50_ms_per_step": float(np.median(step_ms)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "scenes_per_gpu": S, "max_points": 256, "max_tracks": 8,
                       "pose_net": "define_CNN_3D", "pose_dtype": "fp32 (CUDA-core) / bf16x3 split on tcgen05, fp32 accumulate",
                       "dense_path": args.dense_path, "prime_frames": PRIME_FRAMES,
                       "mode": "serial mode: one stream, every kernel of a frame before the next frame's first (what a live "
                               "sensor gets); `throughput_mode` and `e2e` overlap the pose network with the next frame's tracker",
                       "l2": ("NOT flushed (diagnostic run)" if args.no_l2_flush else
                              "flushed between timed steps (256 MiB fill); per-step CUDA events on the library stream, "
                              "flush excluded; steps queued five at a time behind a spin kernel so that host jitter does "
                              "not land inside a step"), "parallelism": "scenes sharded %d/GPU, no collective in the hot loop" % S},
            "throughput_mode": {"value": world * S * K / (tp_ms / 1e3), "unit": UNIT, "ms_per_step": tp_ms / K,
                                "what": "MMW_STEP_PIPELINE: pose network of frame k on a second (high-priority) stream under "
                                        "the tracker of frame k+1, results bit-identical to the serial mode; device-resident "
                                        "inputs, K steps inside one pair of CUDA events, max over ranks",
                                "l2": "no explicit flush (a fill on either stream would serialise them): every step reads a "
                                      "frame never read before and streams ~150 MB through the 126 MB L2"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d // K),
                    "d2h_bytes_per_step": d2h,
                    "api": ("mmw_run_frames" if args.e2e_full_records else "mmw_run_frames_compact") +
                           " (BatchedTracker.run_frames): int16 sensor rows from pinned host memory, throughput mode, " +
                           ("packed result records of every track slot" if args.e2e_full_records else
                            "packed result records of the live tracks (~2 of 8 slots per scene) + their count") +
                           ", every frame, back in pinned host memory",
                    "host": numa,
                    "windows": {"reps": E2E_REPS, "steps_each": K, "value_is": "median over the windows of (steps / max-over-ranks "
                                "wall time)", "scene_frames_per_s": [world * S * K / t for t in e2e_reps]}},
            "gpu_launches": int(launches),
            "latency": latency,
            "clocks": clocks,
            "counters_per_step": {k: float(v) / K for k, v in zip(
                ["scene_frames", "N", "M", "U", "Bf", "tracks", "ring_rows", "pose_rows"], cnt)},
        }
        out.update(rooflines(kern, cnt, K, alg, pk, total_ms / K))
        if world > 1:
            out["multi_gpu_identity"] = identity
        else:
            bt.close()
            del dev
            out["configs"] = other_configs(batches, weights, flush, local)
            out["configs"]["C1"] = {"what": "one scene (what a live 12 Hz sensor sees): host enqueue -> results in host "
                                            "memory, nothing overlapped",
                                    "p50_ms_per_frame": latency.get("p50_ms_single_scene_host_enqueue_to_results")}
        if not args.no_cpu_baseline and world == 1:      # reported at N = 1 only (the reference arm times all host cores)
            from oracle import make_ref
            if make_ref.staged_dir():
                n, sec = reference_run(range(50_000, 50_004), 60)
                out["cpu_baseline"] = {"value": n / sec, "unit": UNIT, "cores": 1, "kind": "reference",
                                       "sample": "4 C2-shaped scenes x 60 frames through the unmodified reference "
                                                 "(oracle/_ref: Utils.normalize_data, TrackBuffer.track, "
                                                 "estimate_posture; filterpy restatement, torch-CPU fp32 pose net "
                                                 "behind .predict), one thread"}
            else:
                n, sec = cpu_port_run(range(50_000, 50_004), 60)
                out["cpu_baseline"] = {"value": n / sec, "unit": UNIT, "cores": 1, "kind": "port",
                                       "sample": "4 C2-shaped scenes x 60 frames, oracle port (numpy float64 + "
                                                 "torch-CPU fp32 pose net), one thread"}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def ncu_traffic():
    """DRAM bytes per launch of each kernel from the committed ncu --set full capture (profiles/r02_traffic.json,
    written by profiles/summarize_ncu.py --traffic), or {} when absent.  STATIC: measured once under the profiler for
    this build, not in this run (a run under ncu is never a bench value)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def issue_roofline(step_ms, traffic):
    """Second roofline of the tracker step: warp instructions per launch (ncu, profiles/r01_traffic.json key
    step_kernel_warp_insts, ~30 k per scene-frame of dependent float64 work) against the issue rate of the chip."""
    wi = traffic.get("step_kernel_warp_insts")
    if not wi:
        return None
    peak = 148 * 4 * 1.965e9            # warp instructions per second at the maximum SM clock
    ach = wi / (step_ms / 1e3)
    return {"bound": "issue", "achieved": ach / 1e9, "peak": peak / 1e9, "unit": "G warp-inst/s", "frac": ach / peak,
            "warp_insts_per_launch": wi,
            "warp_insts_src": "static: ncu smsp__inst_executed.sum of the committed capture (profiles/r02_traffic.json)"}


def rooflines(kern, cnt, K, alg_bytes, pk, step_ms):
    """roofline of the dominant kernel (by CUDA-event time inside the step), plus the two that are always reported:
    the fused tracker step (HBM bound by construction) and the dense-1 GEMM (tensor bound).

    tracker step: algorithmic bytes = SURVEY 8(d) without the pose terms,
        20 N + 4 M + 32 U + 32 Bf[dbscan ran] + sum_tracks 2*624 + 20 * ring rows written + 8 per scene-frame
      (fp32-storage convention of the survey; the device keeps track records in float64, i.e. moves 2x of that term)
    dense 1: algorithmic FLOPs = 2 * rows * 6144 * 1536 (the fp32 layer); the tensor cores execute 3x that
      (bf16x3 split), reported separately as `executed`."""
    out = {}
    frames, N, M, U, Bf, T, ring_rows, rows_total = (float(x) for x in cnt)
    rows = rows_total / K
    fc1_flops = 2.0 * rows * 6144 * 1536
    step_bytes = (20 * N + 4 * M + 32 * U + 32 * Bf + T * 2 * 624 + 20 * ring_rows + 8 * frames) / K
    traffic = ncu_traffic()
    if kern:
        out["kernel_ms"] = kern
        dom = max(kern, key=kern.get)
        st = kern.get("step", None)
        if st:
            a = step_bytes / (st / 1e3) / 1e9
            out["roofline_step"] = {"kernel": "step_kernel", "bound": "hbm", "achieved": a, "peak": pk["hbm_gbs"],
                                    "unit": "GB/s", "frac": a / pk["hbm_gbs"], "traffic": traffic.get("step_kernel"),
                                    "traffic_src": "static: ncu dram bytes of the committed capture (profiles/r02_traffic.json)",
                                    "algorithmic_bytes_per_launch": step_bytes, "peak_src": pk["src"],
                                    # what actually bounds it: warp-instruction issue (ncu smsp__inst_executed.sum of the
                                    # committed capture / (SMs x 4 schedulers x SM clock))
                                    "issue": issue_roofline(st, traffic),
                                    "note": "latency/issue-bound, not HBM-bound: see DESIGN.md section 4 and profiles/"}
        g = kern.get("fc1", None)
        if g:
            a = fc1_flops / (g / 1e3) / 1e12
            out["roofline_fc1"] = {"kernel": "gemm_tc_pair_kernel<176|192|256,3> (dense 1, tcgen05 cta_group::2; tile width picked from the row count)", "bound": "tensor",
                                   "achieved": a,
                                   "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": a / pk["bf16_tflops"],
                                   "traffic": traffic.get("gemm_tc_kernel_dense1"),
                                   "algorithmic_flops_per_launch": fc1_flops, "executed_tflops": 3 * a,
                                   "executed_frac": 3 * a / pk["bf16_tflops"], "peak_src": pk["src"],
                                   "note": "fp32-accurate layer as 3 bf16 MMA passes (hi*hi + hi*lo + lo*hi): "
                                           "`achieved` counts the layer's FLOPs once, `executed` what the tensor "
                                           "pipe ran"}
        cv = kern.get("conv", None)
        if cv:
            # both convolutions of the 3-D net (two launches, timed together): algorithmic FLOPs of the fp32 layers;
            # `executed` = what the MMAs issued (hi/lo split incl. its zero block, 5 -> 8 padded input channels,
            # 256 MMA rows per sample of which 192 are kept)
            conv_flops = 2.0 * rows * (192 * 135 * 16 + 192 * 432 * 32)
            conv_exec = 2.0 * rows * 27 * 256 * (32 * 16 + 64 * 32)
            a = conv_flops / (cv / 1e3) / 1e12
            out["roofline_conv"] = {"kernel": "conv_slab_kernel<16,32,0,3> + conv_slab_kernel<32,64,1,3> (conv 1 + conv 2)",
                                    "bound": "tensor", "achieved": a, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                                    "frac": a / pk["bf16_tflops"], "traffic": traffic.get("conv_slab_conv2"),
                                    "algorithmic_flops_per_launch": conv_flops,
                                    "executed_tflops": conv_exec / (cv / 1e3) / 1e12,
                                    "executed_frac": conv_exec / (cv / 1e3) / 1e12 / pk["bf16_tflops"],
                                    "peak_src": pk["src"],
                                    "note": "shifted-window implicit GEMM, N = 32 / 64 per MMA: bound by the A-operand "
                                            "shared-memory reads of small-N MMAs, not by the tensor pipe (DESIGN.md 4)"}
        by = {"fc1": "roofline_fc1", "conv": "roofline_conv", "step": "roofline_step"}
        out["roofline"] = dict(out.get(by.get(dom, "roofline_step"), out.get("roofline_step", {})))
        out["roofline"]["dominant_kernel"] = dom
        out["algorithmic_bytes_per_step_whole_path"] = alg_bytes / K
    else:
        a = step_bytes / (step_ms / 1e3) / 1e9
        out["roofline"] = {"kernel": "whole step (no per-kernel timing)", "bound": "hbm", "achieved": a,
                           "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": a / pk["hbm_gbs"], "traffic": None}
    return out


if __name__ == "__main__":
    main()
