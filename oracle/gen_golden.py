"""TEST INFRASTRUCTURE ONLY -- regenerates tests/golden/ from the reference itself.

Run in the build container (needs /root/reference, read-only):

    python -m oracle.gen_golden

It executes the reference's own ``Utils.normalize_data``, ``Tracking.TrackBuffer.track``
and ``TrackBuffer.estimate_posture`` (imported unmodified; patches listed in
oracle/ref_harness.py) on seeded synthetic scenes from ``mmwave_msc_b200.synth`` and
stores the per-frame decisions and states, plus the literal known-answer values of
SURVEY.md section 8(c) recomputed from the reference's functions.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mmwave_msc_b200 import synth  # noqa: E402
from oracle import ref_harness as rh, trace_io  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# people walk in and out, clutter confined to a far corner: tracks time out and ids are re-issued
CHURN = synth.SceneSpec(clutter_frac=0.02, leave_prob=0.5, enter_prob=0.5, clutter_box=(2.2, 2.5, 4.2, 4.5),
                        people_min=2, people_max=4)

# (name, scene_id, n_frames, spec, max_tracks)
CASES = [
    ("churn_s311", 311, 150, CHURN, None),
    ("churn_s321", 321, 160, CHURN, None),
    ("churn_s308", 308, 140, CHURN, None),
    ("c1_s0", 0, 60, synth.SceneSpec(), None),
    ("c1_s1", 1, 60, synth.SceneSpec(), None),
    ("c1_s4", 4, 60, synth.SceneSpec(), None),
    ("c1_s5", 5, 60, synth.SceneSpec(), None),
    ("c1_s11", 11, 140, synth.SceneSpec(), None),
    ("c1_s100_long", 100, 200, synth.SceneSpec(), None),
    ("c1_s21_jitter", 21, 40, synth.SceneSpec(jitter_lattice=True), None),
    ("c3_s7_dense", 7, 16, synth.SceneSpec.dense(), 10),
]
# feature maps are stored every 7th frame; the long trace keeps every 14th so that its file stays under 1 MB
FEATURE_EVERY = {"c1_s100_long": 14}


# Clouds built to sit on the edges of the grid screen that the CUDA tracker step puts in front of DBSCAN
# (mmwave_msc_b200/csrc/dbscan.cuh): the reference's own labels, spawns and ids for them.  (name, seed, builder);
# a builder returns the world-frame (x, y', z) blobs of one frame as (n, cx, cy, sigma) tuples plus a clutter count.
SCREEN_CASES = [
    ("screen_outside_grid", 1, lambda h: ([(40, 6.5, 3.0, 0.08)], 0)),             # beyond the 16 cells in x
    ("screen_outside_grid_xy", 2, lambda h: ([(40, -7.0, 11.5, 0.08)], 0)),        # ... in x and y
    ("screen_two_groups", 3, lambda h: ([(20, 0.2, 2.0, 0.03), (20, 0.95, 2.0, 0.03)], 0)),   # one block of cells, out of reach
    ("screen_far_range", 4, lambda h: ([(36, 0.0, 30.0, 0.5)], 0)),                # range weight 0.1: reach 1.7 m
    ("screen_negative_weight", 5, lambda h: ([(36, 0.0, 40.0, 2.0)], 0)),          # weight < 0: everything is a neighbour
    ("screen_cell_corner", 6, lambda h: ([(18, 2 * h - 0.05, 3 * h - 0.05, 0.02), (18, 2 * h + 0.05, 3 * h + 0.05, 0.02)], 0)),
    ("screen_sparse_clutter", 7, lambda h: ([], 90)),                              # many points, nowhere dense
    ("screen_blob_in_clutter", 8, lambda h: ([(30, 1.0, 2.5, 0.1)], 60)),          # 30 < min_samples until the ring fuses
]


def screen_case_frames(seed: int, builder, n_frames: int = 5):
    const, _, _ = rh.load_reference()
    rng = np.random.default_rng(9000 + seed)
    h = float(np.sqrt(const.DB_EPS / (1.0 - const.DB_RANGE_WEIGHT * 3.0)))
    frames = []
    for _ in range(n_frames):
        blobs, n_clutter = builder(h)
        xs, ys, zs = [], [], []
        for n, cx, cy, s in blobs:
            xs.append(rng.normal(cx, s, n)); ys.append(np.abs(rng.normal(cy, s, n)) + 1e-3); zs.append(rng.uniform(0.6, 1.6, n))
        if n_clutter:
            xs.append(rng.uniform(-2.5, 2.5, n_clutter)); ys.append(rng.uniform(0.5, 4.5, n_clutter))
            zs.append(rng.uniform(0.1, 2.4, n_clutter))
        x, yw, zw = np.concatenate(xs), np.concatenate(ys), np.concatenate(zs)
        n = len(x)
        frames.append(synth.raw_from_world(x, yw, zw, rng.choice([0.0, 0.0626, -0.0626, 0.1252], n),
                                           rng.integers(1, 90, n).astype(np.float64), const.S_TILT, const.S_HEIGHT))
    return frames, np.full(n_frames, 0.083)


def known_answers() -> dict:
    const, utils, tracking = rh.load_reference()
    ka = {}
    ka["altered_dist"] = float(utils.altered_EuclideanDist([0.1, 2.0, 1.0], [0.4, 2.5, 0.2]))
    ka["transform"] = utils.point_transform_to_standard_axis(np.array([0.5, 3.0, -0.4, 0.1, 0.6, -0.08])).tolist()
    ka["normalize"] = utils.normalize_data({"x": [.5, 1, 0], "y": [3, -1, 0], "z": [-.4, 0, 0],
                                            "doppler": [.62, .1, .3], "peakVal": [120, 5, 7]}).tolist()
    k = tracking.KalmanState(np.zeros(6))
    k.predict(F=const.MOTION_MODEL.KF_F(0.1), Q=const.MOTION_MODEL.KF_Q_DISCR(0.1))
    ka["predict_diagP_dt0.1"] = np.diag(k.P).tolist()
    ka["Q_dt1"] = const.MOTION_MODEL.KF_Q_DISCR(1).tolist()
    ka["F_dt0.25"] = const.MOTION_MODEL.KF_F(0.25).tolist()
    ka["default_posture"] = np.asarray(const.MODEL_DEFAULT_POSTURE).tolist()
    # row f-2: the reference's own calc_projection_points (Utils.py:180-219); the second input has x_dist == z_dist == 0
    pin = [[1.2, 3.4, 1.1], [0.32, 2.0, 1.3], [-0.7, 1.5, 0.4]]
    ka["projection_points"] = {"inputs": pin, "outputs": [list(map(float, utils.calc_projection_points(*q))) for q in pin]}
    ka["window_constants"] = {n: getattr(const, n) for n in (
        "M_X", "M_Y", "M_Z", "V_SCREEN_FADE_SIZE_MAX", "V_SCREEN_FADE_SIZE_MIN", "V_SCREEN_FADE_WEIGHT")}
    ka["constants"] = {n: getattr(const, n) for n in (
        "S_HEIGHT", "S_TILT", "FB_FRAMES_BATCH", "DB_Z_WEIGHT", "DB_RANGE_WEIGHT", "DB_EPS", "DB_MIN_SAMPLES_MIN",
        "TR_MAX_TRACKS", "TR_LIFETIME_DYNAMIC", "TR_LIFETIME_STATIC", "TR_VEL_THRES", "TR_GATE", "KF_R_STD",
        "KF_Q_STD", "KF_P_INIT", "KF_GROUP_DISP_EST_INIT", "KF_ENABLE_EST", "KF_A_N", "KF_EST_POINTNUM",
        "KF_SPREAD_LIM", "KF_A_SPR", "INTENSITY_MU", "INTENSITY_STD", "MODEL_MIN_INPUT")}
    return ka


def balltree_deviation(n_scenes: int = 24, n_frames: int = 30, first: int = 200, spec=None, max_tracks=None) -> dict:
    """How often the shipped sklearn 'auto' (BallTree) labels differ from exact neighbourhoods."""
    diff_calls = calls = diff_scenes = 0
    for sid in range(first, first + n_scenes):
        sc = synth.gen_scene(sid, n_frames, spec or synth.SceneSpec())
        a = rh.run_reference_scene(sc.frames, sc.dts(), dbscan_algorithm="auto", max_tracks=max_tracks)
        b = rh.run_reference_scene(sc.frames, sc.dts(), dbscan_algorithm="brute", max_tracks=max_tracks)
        sd = False
        for ra, rb in zip(a, b):
            if ra["labels"] is None or rb["labels"] is None:
                sd |= (ra["labels"] is None) != (rb["labels"] is None)
                continue
            calls += 1
            if len(ra["labels"]) != len(rb["labels"]) or not np.array_equal(ra["labels"], rb["labels"]):
                diff_calls += 1
                sd = True
        same_end = ([t["id"] for t in a[-1]["tracks"]] == [t["id"] for t in b[-1]["tracks"]])
        diff_scenes += int(sd or not same_end)
    return {"scenes": n_scenes, "frames": n_frames, "dbscan_calls": calls, "calls_with_different_labels": diff_calls,
            "scenes_with_any_difference": diff_scenes}


def offline_manager_sequence() -> dict:
    """What the reference's CSV reader (Utils.OfflineManager, Utils.py:53-177) hands out frame by frame,
    including its read-buffer quirk: the frame that fills the 40-frame buffer is delivered with its first
    row only (Utils.py:128-131) and the rest of that frame is dropped."""
    import tempfile
    const, utils, tracking = rh.load_reference()
    sc = synth.gen_scene(2, 95)
    d = tempfile.mkdtemp()
    synth.write_reference_csv(sc, d, frames_per_file=40)
    om = utils.OfflineManager(d)
    seq = []
    while not om.is_finished() and len(seq) < 400:
        ok, fc, det = om.get_data()
        seq.append([int(ok), int(fc), len(det["x"]) if ok else -1, int(det["posix"][0]) if ok else -1])
    return {"scene": 2, "frames": 95, "frames_per_file": 40, "sequence": seq}


EXPORT_CASES = [("c1_s4", 4, 30, None), ("churn_s308", None, 140, None)]


def track0_export_golden() -> dict:
    """Row f-3: the dataset-builder export of the reference (its own relative_coordinates + format_batched_frames
    under the loop body of preprocessing.py:185-216) on the frames of two committed traces."""
    out = {}
    for name, _, nf, mt in EXPORT_CASES:
        g = trace_io.unpack(np.load(os.path.join(GOLDEN, name + ".npz")))
        frames, dts = g["frames"][:nf], g["dts"][:nf]
        recs = rh.run_reference_scene(frames, dts, pose_fn=None, max_tracks=mt, export0=True)
        valid = np.array([r["export0"] is not None for r in recs], bool)
        out[name + "_frames"] = np.array(nf, np.int32)
        out[name + "_valid"] = valid
        out[name + "_rows"] = (np.stack([r["export0"][0] for r in recs if r["export0"] is not None])
                               if valid.any() else np.zeros((0, 192, 5)))
        out[name + "_centroid"] = (np.stack([r["export0"][1] for r in recs if r["export0"] is not None])
                                   if valid.any() else np.zeros((0, 2)))
        print("export0", name, "frames", nf, "valid", int(valid.sum()))
    return out


def screen_traces():
    for name, seed, builder in SCREEN_CASES:
        frames, dts = screen_case_frames(seed, builder)
        recs = rh.run_reference_scene(frames, dts, pose_fn=lambda x: np.zeros((len(x), 57)))
        d = trace_io.pack(frames, dts, recs)
        d["max_tracks"] = np.array(4, np.int32)
        np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **d)
        print(name, "frames", len(frames), "tracks at end", len(recs[-1]["tracks"]), "next id", recs[-1]["next_track_id"],
              "dbscan runs", int(d["labels_ran"].sum()),
              "clustered points per run", [int((r["labels"] >= 0).sum()) for r in recs if r["labels"] is not None])


DOPPLER_RES_12HZ = 0.0626302709636043     # dopplerResolutionMps of config_cases/iwr1443sdk2_4m_12hz.cfg (the reference's parser)


def extra_traces():
    """(1) Doppler as the sensor reports it: rows carry dopplerIdx, the reference sees dopplerIdx * dopplerResolutionMps
    in float64 (ReadDataIWR1443.py:163-165) -- values fp32 cannot hold.  (2) a frame without data among the first
    tracked frames: the dataset builder pops the global ring (preprocessing.py:262-264) while it still holds the
    deque's initial empty frame, so the pop removes that and not the first real frame."""
    sc = synth.gen_scene(31, 60)
    idx_frames = []
    for fr in sc.frames:
        r = np.asarray(fr, np.float32).copy()
        r[:, 3] = np.rint(r[:, 3].astype(np.float64) / 0.0626).astype(np.float32)
        idx_frames.append(r)
    g = {"frames": idx_frames, "doppler_res": DOPPLER_RES_12HZ}
    recs = rh.run_reference_scene(trace_io.reference_frames(g), sc.dts(), pose_fn=lambda x: np.zeros((len(x), 57)))
    d = trace_io.pack(idx_frames, sc.dts(), recs, doppler_res=DOPPLER_RES_12HZ)
    d["max_tracks"] = np.array(4, np.int32)
    np.savez_compressed(os.path.join(GOLDEN, "c1_s31_doppler_idx.npz"), **d)
    print("c1_s31_doppler_idx tracks at end", len(recs[-1]["tracks"]), "next id", recs[-1]["next_track_id"])

    # a blob of 22 points per frame: no cluster until two frames are fused (min_samples = 35)
    frames, dts = screen_case_frames(21, lambda h: ([(22, 1.0, 2.5, 0.08)], 40), n_frames=7)
    missing = [False, True, False, False, True, False, False]
    frames = [np.zeros((0, 5), np.float32) if m else f for f, m in zip(frames, missing)]
    recs = rh.run_reference_scene(frames, dts, pose_fn=lambda x: np.zeros((len(x), 57)), missing=missing)
    d = trace_io.pack(frames, dts, recs, missing=missing)
    d["max_tracks"] = np.array(4, np.int32)
    np.savez_compressed(os.path.join(GOLDEN, "ring_pop_placeholder.npz"), **d)
    print("ring_pop_placeholder: ring per frame", [r["ring_counts"].tolist() for r in recs], "tracks",
          [len(r["tracks"]) for r in recs])


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    if "--extra-only" in sys.argv:
        extra_traces()
        return
    if "--screen-only" in sys.argv:
        screen_traces()
        return
    if "--export0-only" in sys.argv:
        np.savez_compressed(os.path.join(GOLDEN, "track0_export.npz"), **track0_export_golden())
        return
    json.dump(offline_manager_sequence(), open(os.path.join(GOLDEN, "offline_manager_sequence.json"), "w"))
    json.dump(known_answers(), open(os.path.join(GOLDEN, "known_answers.json"), "w"), indent=1)
    for name, sid, nf, spec, mt in CASES:
        sc = synth.gen_scene(sid, nf, spec)
        recs = rh.run_reference_scene(sc.frames, sc.dts(), pose_fn=lambda x: np.zeros((len(x), 57)), max_tracks=mt)
        d = trace_io.pack(sc.frames, sc.dts(), recs, feature_every=FEATURE_EVERY.get(name, 7))
        d["max_tracks"] = np.array(4 if mt is None else mt, np.int32)
        trace_io.save_npz(os.path.join(GOLDEN, name + ".npz"), d)
        print(name, "frames", nf, "tracks at end", len(recs[-1]["tracks"]), "next id", recs[-1]["next_track_id"],
              "dbscan runs", int(d["labels_ran"].sum()))
    np.savez_compressed(os.path.join(GOLDEN, "track0_export.npz"), **track0_export_golden())
    screen_traces()
    extra_traces()
    if "--deviation" in sys.argv:
        # C1-like scenes: the residue clouds stay small and the two agree; dense scenes (start-up clouds of hundreds of
        # points per blob): the BallTree prunes true neighbours of the non-metric distance (SURVEY Q2)
        dev = {"c1_like": balltree_deviation(),
               "dense": balltree_deviation(12, 14, 400, synth.SceneSpec.dense(), 10)}
        json.dump(dev, open(os.path.join(GOLDEN, "balltree_deviation.json"), "w"), indent=1)
        print(dev)


if __name__ == "__main__":
    main()
