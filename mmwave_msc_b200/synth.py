"""Seeded synthetic IWR1443-shaped radar sequences (SURVEY.md section 8(d)).

Every scene is generated from its own ``numpy.random.Generator(PCG64(20240 +
scene_id))`` so a scene's frames do not depend on which batch, shard or GPU it
lands on.  Values sit on the lattice the sensor produces
(ReadDataIWR1443.py:118-171 in the reference): x, y, z are multiples of 1/512 m
(int16 / 2**9), Doppler is an integer number of Doppler bins, peakVal is an
integer.  All of them are exactly representable in fp32, so the fp32 buffers
handed to the GPU and the fp64 up-cast handed to the CPU oracle are the same
numbers.

Nothing here touches the device; it only builds host arrays.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Sequence

import numpy as np

S_HEIGHT = 1.8          # reference constants.py:41
S_TILT_DEG = -5.0       # reference constants.py:42


@dataclass
class SceneSpec:
    """Shape of one synthetic workload (defaults: BASELINE config C1/C2)."""
    pts_min: int = 160
    pts_max: int = 240
    people_min: int = 1
    people_max: int = 4
    r_max: float = 4.5              # usable depth of the room [m]
    doppler_res: float = 0.0626     # m/s per Doppler bin (12 Hz cfg)
    frame_ms: int = 83              # 12 Hz
    frame_jitter_ms: int = 2        # +- jitter on the log timestamps
    clutter_frac: float = 0.15
    jitter_lattice: bool = False    # tie-free variant: skip the 1/512 m quantisation (Q21)
    enter_prob: float = 0.1         # fraction of people who walk in late
    leave_prob: float = 0.1         # fraction of people who walk out early (their track must time out)
    clutter_box: tuple = (-2.5, 2.5, 0.3, None)   # x0, x1, y0, y1 (None -> r_max) of the uniform clutter
    t0_ms: int = 1_700_000_000_000
    s_height: float = S_HEIGHT      # mounting of the sensor that sees the scene
    s_tilt_deg: float = S_TILT_DEG

    @staticmethod
    def dense() -> "SceneSpec":
        """BASELINE config C3: 1000 pts/frame, 10 targets, 8.5 m room."""
        return SceneSpec(pts_min=1000, pts_max=1000, people_min=10, people_max=10,
                         r_max=8.5, doppler_res=0.125, frame_ms=100)


@dataclass
class Scene:
    scene_id: int
    frames: List[np.ndarray]        # each (N_f, 5) float32: x, y, z, doppler, peakVal (sensor frame)
    posix_ms: np.ndarray            # (F,) int64 log timestamps
    n_people: int
    people_xy: np.ndarray = field(default=None)  # (F, P, 2) ground truth, world frame

    def dts(self, first_dt: float = 0.1) -> np.ndarray:
        """Per-frame dt exactly as offline_main.py:45-51 computes it."""
        t = self.posix_ms.astype(np.float64) / 1000
        out = np.empty(len(t), dtype=np.float64)
        out[0] = first_dt
        out[1:] = t[1:] - t[:-1]
        return out


def _fold(u: np.ndarray, lo: float, hi: float) -> np.ndarray:
    """Reflect an unbounded walk into [lo, hi] (triangle-wave folding)."""
    w = hi - lo
    v = np.mod(u - lo, 2 * w)
    return lo + np.where(v > w, 2 * w - v, v)


def gen_scene(scene_id: int, n_frames: int, spec: SceneSpec = SceneSpec()) -> Scene:
    """Frames 0..n_frames-1 of scene ``scene_id``.  Prefix-stable: the first k frames do
    not depend on n_frames (each quantity has its own child generator and is drawn
    frame-major)."""
    ss = np.random.SeedSequence(20240 + int(scene_id))
    r_cfg, r_time, r_walk, r_pts = (np.random.Generator(np.random.PCG64(c)) for c in ss.spawn(4))
    P = int(r_cfg.integers(spec.people_min, spec.people_max + 1))
    F = int(n_frames)

    # log timestamps
    step = spec.frame_ms + r_time.integers(-spec.frame_jitter_ms, spec.frame_jitter_ms + 1, size=F)
    posix = spec.t0_ms + np.cumsum(step).astype(np.int64)
    tsec = (posix - posix[0]) / 1000.0

    # people: smooth bounded random walks in the world frame; some enter late / leave early
    p0 = np.stack([r_cfg.uniform(-2.0, 2.0, size=P), r_cfg.uniform(0.8, spec.r_max - 0.3, size=P)], axis=1)
    v0 = r_cfg.uniform(-0.5, 0.5, size=(1, P, 2))
    u = r_cfg.uniform(size=P)
    kind = np.where(u < spec.enter_prob, 0, np.where(u < spec.enter_prob + spec.leave_prob, 1, 2))
    t_evt = r_cfg.integers(15, 120, size=P)
    vel = _fold(np.cumsum(r_walk.normal(0, 0.12, size=(F, P, 2)), axis=0) + v0, -0.7, 0.7)
    dtv = np.diff(tsec, prepend=tsec[0] - spec.frame_ms / 1000.0)[:, None, None]
    walk = p0[None] + np.cumsum(vel * dtv, axis=0)
    pos = np.empty_like(walk)
    pos[..., 0] = _fold(walk[..., 0], -2.5, 2.5)
    pos[..., 1] = _fold(walk[..., 1], 0.5, spec.r_max)
    # effective velocity after reflections
    v_eff = np.empty_like(pos)
    v_eff[1:] = (pos[1:] - pos[:-1]) / dtv[1:]
    v_eff[0] = vel[0]

    th = math.radians(spec.s_tilt_deg)
    c, s = math.cos(th), math.sin(th)
    frames: List[np.ndarray] = []
    for f in range(F):
        present = np.nonzero(np.where(kind == 0, f >= t_evt, np.where(kind == 1, f < t_evt, True)))[0]
        N = int(r_pts.integers(spec.pts_min, spec.pts_max + 1))
        n_cl = int(round(spec.clutter_frac * N))
        n_pp = N - n_cl if len(present) else 0
        N = n_cl + n_pp                      # an empty room only shows clutter (possibly nothing at all)
        owner = present[r_pts.integers(0, max(len(present), 1), size=n_pp)] if n_pp else np.zeros(0, np.int64)
        # world-frame person points
        wx = pos[f, owner, 0] + r_pts.normal(0, 0.12, size=n_pp)
        wy = pos[f, owner, 1] + r_pts.normal(0, 0.12, size=n_pp)
        wz = 1.0 + r_pts.normal(0, 0.40, size=n_pp)
        vx = v_eff[f, owner, 0] + r_pts.normal(0, 0.05, size=n_pp)
        vy = v_eff[f, owner, 1] + r_pts.normal(0, 0.05, size=n_pp)
        # clutter: uniform in the box, random Doppler bins
        cb = spec.clutter_box
        cx = r_pts.uniform(cb[0], cb[1], size=n_cl)
        cy = r_pts.uniform(cb[2], spec.r_max if cb[3] is None else cb[3], size=n_cl)
        cz = r_pts.uniform(0.05, 2.45, size=n_cl)
        X = np.concatenate([wx, cx]); Y = np.concatenate([wy, cy]); Z = np.concatenate([wz, cz])
        # radial velocity seen from the sensor at (0, 0, s_height)
        rx, ry, rz = X, Y, Z - spec.s_height
        rr = np.sqrt(rx * rx + ry * ry + rz * rz) + 1e-9
        dop_p = (vx * rx[:n_pp] + vy * ry[:n_pp]) / rr[:n_pp]
        dop_c = r_pts.normal(0, 0.15, size=n_cl)
        dop = np.concatenate([dop_p, dop_c])
        # world -> sensor frame (inverse of Utils.py:312-327: rotate about X by -tilt after removing the height)
        ys = c * Y + s * (Z - spec.s_height)
        zs = -s * Y + c * (Z - spec.s_height)
        xs = X
        perm = r_pts.permutation(N)          # the sensor does not group points by target
        xs, ys, zs, dop = xs[perm], ys[perm], zs[perm], dop[perm]
        if not spec.jitter_lattice:
            xs = np.round(xs * 512) / 512
            ys = np.round(ys * 512) / 512
            zs = np.round(zs * 512) / 512
        dop = np.round(dop / spec.doppler_res) * spec.doppler_res
        peak = np.floor(r_pts.gamma(0.5, 54.0, size=N)) + 1.0
        fr = np.stack([xs, ys, zs, dop, peak], axis=1).astype(np.float32)
        frames.append(fr)
    return Scene(scene_id=int(scene_id), frames=frames, posix_ms=posix, n_people=P, people_xy=pos)


@dataclass
class FrameBatch:
    """One radar frame of S scenes in the ragged layout the C ABI takes."""
    points: np.ndarray      # (sum N, 5) float32
    offsets: np.ndarray     # (S + 1,) int32
    dt: np.ndarray          # (S,) float64


def gen_batch(scene_ids: Sequence[int], n_frames: int, spec: SceneSpec = SceneSpec(),
              first_dt: float = 0.1) -> List[FrameBatch]:
    """Frames 0..n_frames-1 of the given scenes as per-frame ragged batches."""
    scenes = [gen_scene(s, n_frames, spec) for s in scene_ids]
    dts = np.stack([sc.dts(first_dt) for sc in scenes], axis=0) if scenes else np.zeros((0, n_frames))
    out: List[FrameBatch] = []
    for f in range(n_frames):
        parts = [sc.frames[f] for sc in scenes]
        counts = np.array([p.shape[0] for p in parts], dtype=np.int64)
        offsets = np.zeros(len(parts) + 1, dtype=np.int32)
        offsets[1:] = np.cumsum(counts)
        pts = np.concatenate(parts, axis=0) if parts else np.zeros((0, 5), np.float32)
        out.append(FrameBatch(points=np.ascontiguousarray(pts, dtype=np.float32), offsets=offsets,
                              dt=np.ascontiguousarray(dts[:, f], dtype=np.float64)))
    return out


def raw_from_world(x, yw, zw, doppler, peak, tilt_deg: float = -5.0, height: float = 1.8) -> np.ndarray:
    """Sensor-frame rows (x, y, z, doppler, peakVal; float32) whose world coordinates under the reference's
    transform (Utils.py:312-327: rotation about x by the tilt, then + height) are (x, yw, zw)."""
    th = np.radians(tilt_deg)
    y = np.cos(th) * np.asarray(yw) + np.sin(th) * (np.asarray(zw) - height)
    z = -np.sin(th) * np.asarray(yw) + np.cos(th) * (np.asarray(zw) - height)
    return np.stack([np.asarray(x), y, z, np.asarray(doppler), np.asarray(peak)], axis=1).astype(np.float32)


def write_reference_csv(scene: Scene, directory: str, frames_per_file: int = 200) -> None:
    """Write a scene as a reference experiment log (DataLogging.py:60-89 schema:
    ``frame,x,y,z,doppler,peakVal,posix_ms``; files 1.csv, 2.csv ...; frame numbers
    start at 1 and are consecutive, which is what Utils.py:158-166 relies on)."""
    import os
    os.makedirs(directory, exist_ok=True)
    fidx, fh = 0, None
    for f, fr in enumerate(scene.frames):
        if f % frames_per_file == 0:
            if fh is not None:
                fh.close()
            fidx += 1
            fh = open(os.path.join(directory, f"{fidx}.csv"), "w")
        for row in fr:
            fh.write("%d,%r,%r,%r,%r,%r,%d\n" % (f + 1, float(row[0]), float(row[1]), float(row[2]),
                                                   float(row[3]), float(row[4]), int(scene.posix_ms[f])))
    if fh is not None:
        fh.close()
