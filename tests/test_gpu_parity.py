"""Parity of the CUDA path (called through the C ABI, include/mmw.h) with the numpy oracle and with the
golden traces recorded from the reference.  Decisions (filter, labels, gates, ids) are compared bit-exactly;
float64 state to STATE_RTOL; joints to 1 mm."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from helpers import KEYPOINT_ATOL, STATE_ATOL, STATE_RTOL, compare_frame, oracle_config
from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, default_config
from oracle import mmw_oracle as mo, trace_io

pytestmark = pytest.mark.gpu


# ---- a1: preprocessing --------------------------------------------------------------------------------
def test_preprocess_bit_exact():
    rng = np.random.default_rng(1)
    raw = np.concatenate([synth.gen_scene(3, 4).frames[k] for k in range(4)])
    edge = np.array([[0, 0, 0, .3, 7],            # r == 0 (Utils.py:387-390)
                     [1, -1, 0, .1, 5],           # fails y' > 0
                     [.5, 3, -.4, .62, 120],      # survey known answer
                     [0, 2, 0.8, 0, 1],           # near the z' <= 2.5 bound
                     [0, 1, -2.5, 0, 1]], np.float32)
    rnd = rng.normal(0, 3, size=(5000, 5)).astype(np.float32)
    pts = np.concatenate([raw, edge, rnd]).astype(np.float32)
    bt = BatchedTracker(1)
    world, keep = bt.preprocess(pts)
    ow, ok = mo.normalize_points(pts.astype(np.float64))
    np.testing.assert_array_equal(keep, ok)
    np.testing.assert_array_equal(world[keep], ow)          # bit-exact: same float64 operations, no FMA contraction


# ---- a2/a3: DBSCAN ------------------------------------------------------------------------------------
def test_dbscan_stage_matches_oracle():
    rng = np.random.default_rng(2)
    clouds = []
    for n, k in ((0, 1), (1, 1), (34, 1), (35, 1), (90, 2), (400, 3), (600, 4), (768, 5)):
        c = np.concatenate([rng.normal([rng.uniform(-2, 2), rng.uniform(1, 4), 1.0], [0.12, 0.12, 0.4],
                                       size=(n // k if k else 0, 3)) for _ in range(k)] +
                           [rng.uniform([-2.5, 0.3, 0], [2.5, 4.5, 2.5], size=(n - (n // k) * k, 3))]) if n else \
            np.zeros((0, 3))
        clouds.append(c)
    # a cloud that mixes dense blobs and uniform clutter
    clouds.append(np.concatenate([rng.normal([0, 2, 1], [0.12, 0.12, 0.4], size=(150, 3)),
                                  rng.uniform([-2.5, 0.3, 0], [2.5, 4.5, 2.5], size=(300, 3))]))
    bt = BatchedTracker(1, max_points=256)
    got = bt.dbscan(clouds)
    for c, g in zip(clouds, got):
        pts8 = np.zeros((len(c), 8)); pts8[:, :3] = c
        np.testing.assert_array_equal(g, mo.dbscan_labels(pts8))
    # border/tie semantics on the hand-made cloud of the oracle test
    p = np.zeros((10, 3)); p[:, 0] = [0.35, 0.55, 0.6, 0.65, 0.7, 0.0, 0.05, 0.1, 0.15, 5.0]
    assert bt.dbscan([p], eps=0.05, min_samples=4)[0].tolist() == [0, 0, 0, 0, 0, 1, 1, 1, 1, -1]


# ---- a6/a7: Kalman ------------------------------------------------------------------------------------
def _rand_spd(rng, n, scale=0.1):
    a = rng.normal(size=(n, n))
    return scale * (a @ a.T / n + np.eye(n))


def test_kalman_predict_update_stage():
    rng = np.random.default_rng(3)
    n = 37
    x = rng.normal(size=(n, 9)); P = np.stack([_rand_spd(rng, 9) for _ in range(n)])
    dt = rng.uniform(0.05, 3.5, size=n)
    bt = BatchedTracker(1)
    gx, gP = bt.kalman_predict(x, P, dt)
    for i in range(n):
        F, Q = mo.kf_F(dt[i]), mo.kf_Q(dt[i])
        np.testing.assert_allclose(gx[i], F @ x[i], rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(gP[i], (F @ P[i]) @ F.T + Q, rtol=1e-13, atol=1e-15)
    z = rng.normal(size=(n, 6)); R = np.stack([_rand_spd(rng, 6, 0.01) for _ in range(n)])
    life0 = rng.integers(0, 2, size=n).astype(np.uint8)
    ux, uP = bt.kalman_update(x, P, z, R, life0)
    cfg = mo.OracleConfig()
    for i in range(n):
        t = mo.Track(np.zeros((1, 8)), 0, cfg)
        t.x, t.P, t.centroid, t.lifetime = x[i].copy(), P[i].copy(), z[i], 0.0 if life0[i] else 0.5
        t.Rc = lambda R_=R[i]: R_
        t.update()
        np.testing.assert_allclose(ux[i], t.x, rtol=1e-11, atol=1e-13)
        np.testing.assert_allclose(uP[i], t.P, rtol=1e-10, atol=1e-13)


def test_gate_stage():
    rng = np.random.default_rng(4)
    T, M = 5, 300
    hx = rng.normal(0, 1, size=(T, 6)); Cm = np.stack([_rand_spd(rng, 6, 0.3) for _ in range(T)])
    pts = hx[rng.integers(0, T, size=M)] + rng.normal(0, 0.6, size=(M, 6))
    bt = BatchedTracker(1)
    d2, assoc = bt.gate(pts, hx, Cm)
    ref = np.stack([np.log(abs(np.linalg.det(Cm[j]))) + np.einsum("ia,ab,ib->i", pts - hx[j], np.linalg.inv(Cm[j]),
                                                                  pts - hx[j]) for j in range(T)], axis=1)
    np.testing.assert_allclose(d2, ref, rtol=1e-11, atol=1e-12)
    exp = mo.associate_from_scores(ref, 4.5)
    margin = np.abs(ref - 4.5).min(axis=1)
    assert np.array_equal(assoc[margin > 1e-9], exp[margin > 1e-9])
    assert (assoc >= 0).sum() > 20 and (assoc < 0).sum() > 20


# ---- a15/a16: pose CNN --------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [pw.VARIANT_3D, pw.VARIANT_2D])
@pytest.mark.parametrize("tensor_cores", [False, True])
def test_pose_stage(variant, tensor_cores):
    rng = np.random.default_rng(5)
    fb = 2 if variant == pw.VARIANT_3D else 0
    W = pw.make_pose_weights(variant)
    n = 200
    shape = (n, 3, 8, 8, 5) if fb == 2 else (n, 8, 8, 5)
    feats = np.zeros((n, (fb + 1) * 64, 5), np.float32)
    for i in range(n):                       # 20-64 real rows per frame + zero pads, like format_single_frame
        for f in range(fb + 1):
            k = int(rng.integers(20, 65))
            rows = np.zeros((64, 5), np.float32)
            rows[:k, 0] = rng.normal(0, 0.15, k); rows[:k, 1] = rng.normal(0, 0.15, k)
            rows[:k, 2] = rng.normal(1.0, 0.4, k); rows[:k, 3] = rng.normal(0, 0.3, k)
            rows[:k, 4] = (np.floor(rng.gamma(0.5, 54.0, k)) + 1 - 27.0187) / 70.351
            feats[i, f * 64:(f + 1) * 64] = rows[np.argsort(rows[:, 0], kind="stable")]
    feats = feats.reshape(shape)
    bt = BatchedTracker(64, max_tracks=8, config=default_config(frames_batch=fb))
    bt.load_pose_weights(W, variant)
    bt.set_dense_path(tensor_cores)
    got = bt.pose(feats)
    ref = mo.pose_forward(W, feats, np.float64)
    err = np.abs(got - ref).max()
    assert err < (KEYPOINT_ATOL if tensor_cores else 1e-4), "max joint error %.3g m" % err
    assert np.abs(ref).mean() > 0.05         # the comparison is not vacuous


# ---- a11: full sequences, free-running ----------------------------------------------------------------
def _run_sequence(scene_ids, n_frames, spec, cfg, weights=None, tensor_cores=True, max_points=256, max_tracks=8,
                  every=1):
    batches = synth.gen_batch(scene_ids, n_frames, spec)
    ocfg = oracle_config(cfg)
    oracles = [mo.SceneOracle(ocfg, pose_weights=weights, pose_dtype=np.float64) for _ in scene_ids]
    bt = BatchedTracker(len(scene_ids), max_points=max_points, max_tracks=max_tracks, config=cfg)
    if weights is not None:
        bt.load_pose_weights(weights)
        bt.set_dense_path(tensor_cores)
    for f, b in enumerate(batches):
        bt.step(b.points, b.offsets, b.dt, pose=weights is not None, record_labels=True)
        recs = [o.step(b.points[b.offsets[s]:b.offsets[s + 1]], b.dt[s]) for s, o in enumerate(oracles)]
        if f % every == 0 or f == n_frames - 1:
            compare_frame(bt, recs, b.offsets, "frame %d" % f, labels=bt.labels(),
                          check_keypoints=weights is not None,
                          pose_rows=bt.pose_rows() if weights is not None else None)
    assert not bt.status().any()
    return bt


def test_sequences_default_config_with_pose():
    W = pw.make_pose_weights(pw.VARIANT_3D)
    _run_sequence(list(range(12)), 45, synth.SceneSpec(), default_config(), weights=W)


def test_feature_sort_lattice_fast_path_and_exact_path(monkeypatch):
    """pose_feature_kernel ranks the 64 rows of a frame by (x - cx, index).  On the sensor's lattice (x a multiple of
    2^-16) it compares 32-bit integer images of x; otherwise the order-preserving int64 images of the float64 keys.
    Both must give the reference's order: the exact path on off-lattice inputs against the oracle, and both paths
    bit-identical on lattice inputs."""
    W = pw.make_pose_weights(pw.VARIANT_3D)
    ids, nf = [3, 4, 9, 11], 16
    # (1) off-lattice x (fp32 values that are not multiples of 2^-16): the exact path, checked against the oracle
    batches = synth.gen_batch(ids, nf, synth.SceneSpec())
    rng = np.random.default_rng(17)
    for b in batches:
        b.points[:, 0] = (b.points[:, 0].astype(np.float64) + rng.uniform(-3e-6, 3e-6, len(b.points))).astype(np.float32)
    assert (np.rint(batches[3].points[:, 0].astype(np.float64) * 65536) != batches[3].points[:, 0].astype(np.float64) * 65536).any()
    cfg = default_config()
    oracles = [mo.SceneOracle(oracle_config(cfg), pose_weights=W, pose_dtype=np.float64) for _ in ids]
    bt = BatchedTracker(len(ids), config=cfg)
    bt.load_pose_weights(W)
    for f, b in enumerate(batches):
        bt.step(b.points, b.offsets, b.dt, pose=True, record_labels=True)
        recs = [o.step(b.points[b.offsets[s]:b.offsets[s + 1]], b.dt[s]) for s, o in enumerate(oracles)]
        compare_frame(bt, recs, b.offsets, "off-lattice frame %d" % f, labels=bt.labels(), check_keypoints=True,
                      pose_rows=bt.pose_rows())
    bt.close()
    # (2) lattice inputs: fast path == exact path, bit for bit (feature maps and keypoints)
    batches = synth.gen_batch(ids, nf, synth.SceneSpec())
    runs = []
    for dbg in ("0", "16"):
        monkeypatch.setenv("MMW_FEAT_DBG", dbg)
        bt = BatchedTracker(len(ids), config=cfg)
        bt.load_pose_weights(W)
        out = []
        for b in batches:
            bt.step(b.points, b.offsets, b.dt, pose=True)
            si, ti, feats = bt.pose_rows()
            out.append((si.copy(), ti.copy(), feats.copy(), bt.tracks()[0].tobytes()))
        runs.append(out)
        bt.close()
    monkeypatch.delenv("MMW_FEAT_DBG")
    assert sum(len(o[0]) for o in runs[0]) > 3 * nf
    for a, b in zip(*runs):
        for u, v in zip(a, b):
            assert u == v if isinstance(u, bytes) else np.array_equal(u, v)


def test_sequences_churn_tracks_time_out_and_ids_reissued():
    spec = synth.SceneSpec(clutter_frac=0.02, leave_prob=0.5, enter_prob=0.5, clutter_box=(2.2, 2.5, 4.2, 4.5),
                           people_min=2, people_max=4)
    bt = _run_sequence([304, 308, 311, 321], 150, spec, default_config())
    _, nid, _ = bt.summary()
    _, nt = bt.tracks()
    assert (nid > nt).any()                   # at least one track was dropped


def test_sequences_2d_net_frames_batch_0():
    W = pw.make_pose_weights(pw.VARIANT_2D)
    _run_sequence([1, 2, 5], 25, synth.SceneSpec(), default_config(frames_batch=0), weights=W)


def test_sequence_dense_config_c3():
    _run_sequence([7, 8], 10, synth.SceneSpec.dense(), default_config(tr_max_tracks=10), max_points=1024,
                  max_tracks=16)


def test_empty_and_ragged_frames():
    """Scenes with no points at all, frames emptied by the filter (Q23), and a scene that only ever sees noise."""
    cfg = default_config()
    bt = BatchedTracker(4, config=cfg)
    oracles = [mo.SceneOracle(oracle_config(cfg)) for _ in range(4)]
    sc = synth.gen_scene(1, 12)
    rng = np.random.default_rng(9)
    for f in range(12):
        parts = [sc.frames[f],
                 np.zeros((0, 5), np.float32),                                             # empty input
                 np.array([[1, -1, 0, .1, 5], [0, 0, 0, .2, 3]], np.float32),              # all filtered out
                 rng.uniform([-2, 0.5, -1, -1, 1], [2, 4, 0.5, 1, 50], size=(int(rng.integers(1, 40)), 5)).astype(
                     np.float32)]
        if f % 5 == 4:
            parts[0] = np.zeros((0, 5), np.float32)                                        # a dropped frame
        offsets = np.zeros(5, np.int32); offsets[1:] = np.cumsum([len(p) for p in parts])
        pts = np.concatenate(parts)
        dt = np.full(4, 0.083)
        bt.step(pts, offsets, dt, pose=False, record_labels=True)
        recs = [o.step(p, 0.083) for o, p in zip(oracles, parts)]
        compare_frame(bt, recs, offsets, "frame %d" % f, labels=bt.labels())


def _raw_from_world(x, yw, zw, doppler, peak, cfg):
    """Sensor-frame rows whose world coordinates (Utils.py:312-327) are (x, yw, zw)."""
    th = np.radians(cfg.s_tilt_deg)
    y = np.cos(th) * yw + np.sin(th) * (zw - cfg.s_height)
    z = -np.sin(th) * yw + np.cos(th) * (zw - cfg.s_height)
    return np.stack([x, y, z, doppler, peak], axis=1).astype(np.float32)


def test_grid_screen_edge_cases():
    """The step kernel decides 'no point can be a core point' on a clamped 16 x 16 grid over (x, y') before it counts
    neighbours (dbscan.cuh).  Clouds built to sit on the edges of that screen -- blobs outside the grid, on cell
    borders, one point short of min_samples, far range where the range weight widens the reach, range beyond which
    the weight turns negative -- must give the oracle's labels, spawns and ids."""
    cfg = default_config()
    rng = np.random.default_rng(77)

    def blob(n, cx, cy, sx, sy):
        return _raw_from_world(rng.normal(cx, sx, n), rng.normal(cy, sy, n), rng.uniform(0.6, 1.6, n),
                               rng.choice([0.0, 0.0626, -0.0626], n), rng.integers(1, 90, n).astype(np.float64), cfg)

    def clutter(n):
        return _raw_from_world(rng.uniform(-2.5, 2.5, n), rng.uniform(0.5, 4.5, n), rng.uniform(0.1, 2.4, n),
                               rng.choice([0.0, 0.0626, -0.125], n), rng.integers(1, 60, n).astype(np.float64), cfg)

    h = float(np.sqrt(cfg.db_eps / (1.0 - cfg.db_range_weight * 3.0)))      # about one grid cell at 3 m
    makers = [
        lambda f: blob(40, 6.5, 3.0, 0.08, 0.08),                             # beyond the grid in x (folded onto its border)
        lambda f: blob(40, -7.0, 11.5, 0.08, 0.08),                           # beyond it in x and y
        lambda f: np.concatenate([blob(20, 0.2, 2.0, 0.03, 0.03), blob(20, 0.95, 2.0, 0.03, 0.03)]),   # 40 points in one
        #   block of cells but two groups out of each other's reach: screened in, no core point until the ring fuses two frames
        lambda f: blob(36, 0.0, 30.0, 0.5, 0.5),                              # far range: reach sqrt(eps / 0.1) = 1.7 m
        lambda f: blob(36, 0.0, 40.0, 2.0, 2.0),                              # range weight negative: everything is a neighbour
        lambda f: np.concatenate([blob(18, 2 * h - 0.05, 3 * h - 0.05, 0.02, 0.02),
                                  blob(18, 2 * h + 0.05, 3 * h + 0.05, 0.02, 0.02)]),   # one blob straddling a cell corner
        lambda f: clutter(20),                                                # never reaches min_samples points at all
        lambda f: clutter(90),                                                # plenty of points, nowhere dense
    ]
    S = len(makers)
    bt = BatchedTracker(S, config=cfg)
    oracles = [mo.SceneOracle(oracle_config(cfg)) for _ in range(S)]
    spawned = np.zeros(S, bool)
    for f in range(5):
        parts = [m(f) for m in makers]
        offsets = np.zeros(S + 1, np.int32); offsets[1:] = np.cumsum([len(p) for p in parts])
        dt = np.full(S, 0.083)
        bt.step(np.concatenate(parts), offsets, dt, pose=False, record_labels=True)
        recs = [o.step(p, 0.083) for o, p in zip(oracles, parts)]
        compare_frame(bt, recs, offsets, "frame %d" % f, labels=bt.labels())
        spawned |= np.array([len(r["tracks"]) > 0 for r in recs])
    assert spawned[[0, 1, 2, 3, 4, 5]].all() and not spawned[[6, 7]].any()    # both outcomes were exercised
    assert not bt.status().any()


# ---- golden traces recorded from the reference's own Tracking.py / Utils.py --------------------------
@pytest.mark.parametrize("case", golden_cases())
def test_against_reference_golden_trace(case):
    d = np.load(os.path.join(GOLDEN, case + ".npz"))
    g = trace_io.unpack(d)
    mt = int(d["max_tracks"])
    dense = max(len(f) for f in g["frames"]) > 256
    # rows as the sensor reports them: the Doppler column in units of doppler_res (c1_s31_doppler_idx: the index)
    bt = BatchedTracker(1, max_points=1024 if dense else 256, max_tracks=16 if dense else 8,
                        config=default_config(tr_max_tracks=mt, doppler_res=g["doppler_res"]))
    bt.load_pose_weights(pw.make_pose_weights(pw.VARIANT_3D))
    for f, (fr, dt, rec) in enumerate(zip(g["frames"], g["dts"], g["recs"])):
        offsets = np.array([0, len(fr)], np.int32)
        if g["missing"][f]:
            bt.ring_pop(0)                               # a frame without data (preprocessing.py:262-264)
        want_pose = rec["features"] is not None
        bt.step(fr, offsets, np.array([dt]), pose=want_pose, record_labels=True)
        compare_frame(bt, [rec], offsets, "%s frame %d" % (case, f), labels=bt.labels(),
                      pose_rows=bt.pose_rows() if want_pose else None)


# ---- size-independent properties at the benchmark's full size ----------------------------------------
def test_full_size_c2_permutation_and_determinism():
    S, F = 1024, 6
    ids = list(range(S))
    batches = synth.gen_batch(ids, F)
    W = pw.make_pose_weights(pw.VARIANT_3D)

    def run(order):
        bt = BatchedTracker(S)
        bt.load_pose_weights(W)
        for b in batches:
            parts = [b.points[b.offsets[s]:b.offsets[s + 1]] for s in order]
            offsets = np.zeros(S + 1, np.int32); offsets[1:] = np.cumsum([len(p) for p in parts])
            bt.step(np.concatenate(parts), offsets, b.dt[order], pose=True)
        tr, nt = bt.tracks()
        return tr, nt, bt.status()

    ident = np.arange(S)
    perm = np.random.default_rng(0).permutation(S)
    tr0, nt0, st0 = run(ident)
    tr1, nt1, _ = run(ident)
    trp, ntp, _ = run(perm)
    assert not st0.any()
    assert nt0.sum() > S                       # tracks exist
    assert tr0.tobytes() == tr1.tobytes()      # run-to-run bit-identical
    inv = np.argsort(perm)
    assert np.array_equal(nt0, ntp[inv])
    assert tr0.tobytes() == trp[inv].tobytes() # a scene's result does not depend on its place in the batch
    # spot-check 8 scenes against the oracle
    pick = [0, 17, 233, 511, 512, 640, 901, 1023]
    oracles = {s: mo.SceneOracle(pose_weights=W) for s in pick}
    for b in batches:
        recs = {s: oracles[s].step(b.points[b.offsets[s]:b.offsets[s + 1]], b.dt[s]) for s in pick}
    for s in pick:
        assert nt0[s] == len(recs[s]["tracks"])
        for k, t in enumerate(recs[s]["tracks"]):
            assert tr0[s, k]["id"] == t["id"]
            np.testing.assert_allclose(tr0[s, k]["x"], t["x"], rtol=1e-8, atol=1e-10)
            np.testing.assert_allclose(tr0[s, k]["keypoints"], t["keypoints"], rtol=0, atol=KEYPOINT_ATOL)


# ---- pipelined host path: side-stream upload + asynchronous packed-result download -----------------
def _tiled(batches, reps):
    """reps copies of the generated scenes side by side: scene s + k * S is scene s again."""
    out = []
    for b in batches:
        n = b.points.shape[0]
        off = np.concatenate([b.offsets[:-1] + k * n for k in range(reps)] + [np.array([reps * n], np.int32)])
        out.append((np.tile(b.points, (reps, 1)), off.astype(np.int32), np.tile(b.dt, reps)))
    return out


def _spot_check_against_oracle(bt, tiled, gen_batches, S_gen, pick, ocfg, W, every=4):
    """Scenes `pick` of the big batch (each a copy of generated scene pick % S_gen) against the oracle, every few
    frames: track count, ids, association of every point, Kalman state; keypoints at the end."""
    oracles = {s: mo.SceneOracle(ocfg, pose_weights=W) for s in pick}
    F = len(tiled)
    for f, (pts, off, dt) in enumerate(tiled):
        bt.step(pts, off, dt, pose=W is not None)
        b = gen_batches[f]
        recs = {s: oracles[s].step(b.points[b.offsets[s % S_gen]:b.offsets[s % S_gen + 1]], b.dt[s % S_gen]) for s in pick}
        if f % every and f != F - 1:
            continue
        tr, nt = bt.tracks()
        assoc = bt.point_assoc()
        for s in pick:
            r = recs[s]
            ctx = "frame %d scene %d" % (f, s)
            assert nt[s] == len(r["tracks"]), ctx
            np.testing.assert_array_equal(assoc[off[s]:off[s] + r["M"]], r["assoc"], err_msg=ctx)
            for k, t in enumerate(r["tracks"]):
                assert tr[s, k]["id"] == t["id"] and tr[s, k]["point_num"] == t["point_num"], ctx
                np.testing.assert_allclose(tr[s, k]["x"], t["x"], rtol=STATE_RTOL, atol=STATE_ATOL, err_msg=ctx)
                np.testing.assert_allclose(tr[s, k]["P"], t["P"], rtol=STATE_RTOL, atol=STATE_ATOL, err_msg=ctx)
                if W is not None and f == F - 1:
                    np.testing.assert_allclose(tr[s, k]["keypoints"], t["keypoints"], rtol=0, atol=KEYPOINT_ATOL,
                                               err_msg=ctx)
    return nt


def test_full_size_c5_8192_scenes_on_one_gpu_oracle_spot_checks():
    """BASELINE config C5 on one GPU: 8192 scenes in one context (the pose-row scan takes its separate kernel above
    4096 scenes), 36 scenes spread over the batch against the oracle for 20 frames, and the eight copies of every
    generated scene agree bit for bit."""
    S_gen, reps, F = 1024, 8, 20
    gen = synth.gen_batch(list(range(3000, 3000 + S_gen)), F)
    tiled = _tiled(gen, reps)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    bt = BatchedTracker(S_gen * reps)
    bt.load_pose_weights(W)
    pick = sorted(set(int(x) for x in np.random.default_rng(5).integers(0, S_gen * reps, 34)) | {0, 8191})
    nt = _spot_check_against_oracle(bt, tiled, gen, S_gen, pick, mo.OracleConfig(), W)
    assert not bt.status().any() and nt.sum() > S_gen * reps
    tr, nt = bt.tracks()
    tr = tr.reshape(reps, S_gen, -1)
    for k in range(1, reps):
        assert tr[0].tobytes() == tr[k].tobytes()
    bt.close()


def test_full_size_c3_dense_1024_scenes_oracle_spot_checks():
    """BASELINE config C3 at 1024 scenes: 1000 points per frame, 10 targets, TR_MAX_TRACKS = 10 (fused clouds of up to
    3000 points: the large-cloud DBSCAN path), 12 scenes against the oracle for 10 frames."""
    S_gen, reps, F = 256, 4, 10
    gen = synth.gen_batch(list(range(5000, 5000 + S_gen)), F, synth.SceneSpec.dense())
    tiled = _tiled(gen, reps)
    cfg = default_config(tr_max_tracks=10)
    bt = BatchedTracker(S_gen * reps, max_points=1024, max_tracks=16, config=cfg)
    pick = sorted(set(int(x) for x in np.random.default_rng(7).integers(0, S_gen * reps, 10)) | {0, 1023})
    nt = _spot_check_against_oracle(bt, tiled, gen, S_gen, pick, oracle_config(cfg), None, every=3)
    assert not bt.status().any() and nt.mean() > 3
    bt.close()


def test_pipelined_results_match_blocking_readback():
    import torch
    S, F = 64, 10
    batches = synth.gen_batch(list(range(S)), F)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    bt = BatchedTracker(S)
    bt.load_pose_weights(W)
    ref = BatchedTracker(S)
    ref.load_pose_weights(W)
    host = [torch.empty(S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32).pin_memory().numpy() for _ in range(2)]
    pinned = []
    for b in batches:                      # the API keeps reading the caller's buffers until the copy has run
        pinned.append((torch.from_numpy(b.points).pin_memory().numpy(), torch.from_numpy(b.offsets).pin_memory().numpy(),
                       torch.from_numpy(b.dt).pin_memory().numpy()))
    prev = None
    snaps = []
    for f, (p, o, d) in enumerate(pinned):
        bt.step(p, o, d, pose=True)
        slot = bt.read_results_async(host[f & 1])
        if prev is not None:
            bt.wait_results(prev[0])
            snaps.append(host[prev[1]].copy())
        prev = (slot, f & 1)
    bt.wait_results(prev[0])
    snaps.append(host[prev[1]].copy())
    for f, b in enumerate(batches):
        ref.step(b.points, b.offsets, b.dt, pose=True)
        tr, nt = ref.tracks()
        got = snaps[f].reshape(S, bt.tcap, _lib.RESULT_FLOATS)
        for s in range(S):
            assert int(got[s, 0, 1]) == nt[s]
            for k in range(nt[s]):
                assert int(got[s, k, 0]) == tr[s, k]["id"]
                np.testing.assert_array_equal(got[s, k, 2:11], tr[s, k]["x"].astype(np.float32))
                np.testing.assert_array_equal(got[s, k, 11:68], tr[s, k]["keypoints"])
                # row f-2: fade square of the smart window, float64 on both sides, stored as fp32
                (cx, cz), size = mo.fade_square(tr[s, k]["x"], tr[s, k]["keypoints"])
                np.testing.assert_array_equal(got[s, k, 68:71], np.array([cx, cz, size]).astype(np.float32))
            assert np.all(got[s, nt[s]:, 0] == -1)


# ---- alternative code paths selected by environment switches give the same results -------------------------
def _run_with_env(env, S=48, F=14):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        batches = synth.gen_batch(list(range(100, 100 + S)), F)
        bt = BatchedTracker(S)                                  # MMW_POSE_INDEX_FOLD is read at creation,
        bt.load_pose_weights(pw.make_pose_weights(pw.VARIANT_3D))   # MMW_FC1_BN when the weights are loaded
        for b in batches:
            bt.step(b.points, b.offsets, b.dt, pose=True)
        tr, nt = bt.tracks()
        si, ti, feats = bt.pose_rows()
        return tr, nt, si, ti, feats
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_throughput_mode_results_are_bit_identical_to_serial_mode():
    """MMW_STEP_PIPELINE: the pose network of frame k on its own stream under the tracker of frame k + 1.  The packed
    records fetched per frame equal the serial mode's bit for bit -- also for scenes whose frame is skipped (their
    tracks get no pose row) and across a switch back to the serial mode; the final track records agree too."""
    S, F = 48, 30
    batches = synth.gen_batch(list(range(700, 700 + S)), F)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    n = S * 8 * _lib.RESULT_FLOATS
    a, b = BatchedTracker(S), BatchedTracker(S)
    a.load_pose_weights(W); b.load_pose_weights(W)
    rng = np.random.default_rng(3)
    out_a = [np.zeros(n, np.float32) for _ in range(F)]
    out_b = [np.zeros(n, np.float32) for _ in range(F)]
    slots = []
    for f, bt in enumerate(batches):
        pts, off, dt = bt.points, bt.offsets, bt.dt
        if f in (9, 10, 17):                                     # a few scenes lose their frame (Q23)
            drop = rng.choice(S, 5, replace=False)
            parts = [pts[off[s]:off[s + 1]] if s not in drop else pts[:0] for s in range(S)]
            pts = np.concatenate(parts); off = np.zeros(S + 1, np.int32); off[1:] = np.cumsum([len(p) for p in parts])
        serial_here = f in (20, 21)                              # mode switch in the middle of the sequence
        a.step(pts, off, dt, pose=True)
        a.wait_results(a.read_results_async(out_a[f]))
        b.step(pts, off, dt, pose=True, pipeline=not serial_here)
        slots.append(b.read_results_async(out_b[f]))
        if f >= 1:
            b.wait_results(slots[f - 1])
    b.wait_results(slots[-1])
    for f in range(F):
        assert out_a[f].tobytes() == out_b[f].tobytes(), "frame %d" % f
    ta, na = a.tracks()
    tb, nb = b.tracks()
    assert na.sum() > S and np.array_equal(na, nb) and ta.tobytes() == tb.tobytes()


def test_int16_lattice_input_and_run_frames_equal_the_fp32_path():
    """MMW_STEP_INPUT_I16: rows as the sensor reports them (int16 x, y, z in Q9, dopplerIdx, peakVal; 10 bytes per
    point) give bit for bit what the fp32 rows of the same lattice values give; mmw_run_frames (the replay loop in C,
    throughput mode) gives what stepping frame by frame gives."""
    S, F, RES = 24, 18, 0.0626302709636043      # 18 frames: run_frames uploads them in groups of 4 + a group of 2
    batches = synth.gen_batch(list(range(900, 900 + S)), F)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    cfg = default_config(doppler_res=RES, xyz_q_format=9)
    f32, i16 = [], []
    for b in batches:
        p = b.points.astype(np.float64)
        q = np.stack([np.rint(p[:, 0] * 512), np.rint(p[:, 1] * 512), np.rint(p[:, 2] * 512), np.rint(p[:, 3] / 0.0626),
                      p[:, 4]], axis=1)
        assert np.array_equal(q[:, :3] / 512, p[:, :3]) and np.abs(q).max() < 32768
        i16.append(np.ascontiguousarray(q.astype(np.int16)))
        f32.append(np.ascontiguousarray(np.stack([q[:, 0] / 512, q[:, 1] / 512, q[:, 2] / 512, q[:, 3], q[:, 4]], 1).astype(np.float32)))
    n = S * 8 * _lib.RESULT_FLOATS
    a, b_, c_ = BatchedTracker(S, config=cfg), BatchedTracker(S, config=cfg), BatchedTracker(S, config=cfg)
    for t in (a, b_, c_):
        t.load_pose_weights(W)
    ra, rb = np.zeros((F, n), np.float32), np.zeros((F, n), np.float32)
    for f, bt in enumerate(batches):
        a.step(f32[f], bt.offsets, bt.dt, pose=True)
        a.wait_results(a.read_results_async(ra[f]))
        b_.step(i16[f], bt.offsets, bt.dt, pose=True)
        b_.wait_results(b_.read_results_async(rb[f]))
    assert ra.tobytes() == rb.tobytes()
    ta, na = a.tracks(); tb, nb = b_.tracks()
    assert na.sum() > S and ta.tobytes() == tb.tobytes()
    rc = np.zeros((F, n), np.float32)
    rows = np.concatenate(i16)
    fro = np.cumsum([0] + [len(x) for x in i16]).astype(np.int64)
    c_.run_frames(rows, fro, np.stack([bt.offsets for bt in batches]), np.stack([bt.dt for bt in batches]), rc)
    assert rc.tobytes() == ra.tobytes()
    # mmw_run_frames_compact: only the live tracks' records come back (written by a kernel into pinned host memory);
    # expanded again they are the full records, bit for bit -- in throughput mode and in serial mode
    import torch
    for pipeline in (True, False):
        d_ = BatchedTracker(S, config=cfg)
        d_.load_pose_weights(W)
        rd = torch.zeros((F, n), dtype=torch.float32).pin_memory().numpy()
        cnt = torch.zeros(F, dtype=torch.int32).pin_memory().numpy()
        d_.run_frames(rows, fro, np.stack([bt.offsets for bt in batches]), np.stack([bt.dt for bt in batches]), rd,
                      pipeline=pipeline, n_records=cnt)
        assert cnt[-1] == na.sum() and (cnt[2:] > 0).all()
        for f in range(F):
            full = d_.expand_compact_results(rd[f], int(cnt[f]))
            assert full.tobytes() == ra[f].tobytes(), "frame %d" % f
        d_.close()
    with pytest.raises(_lib.MmwError):         # pageable host memory is refused, not silently staged
        e_ = BatchedTracker(S, config=cfg)
        e_.load_pose_weights(W)
        e_.run_frames(rows, fro, np.stack([bt.offsets for bt in batches]), np.stack([bt.dt for bt in batches]),
                      np.zeros((F, n), np.float32), n_records=np.zeros(F, np.int32))
    # ... and against the oracle on the float64 values the lattice stands for
    so = mo.SceneOracle(pose_weights=W)
    for f, bt in enumerate(batches):
        fr = f32[f][bt.offsets[3]:bt.offsets[4]].astype(np.float64)
        fr[:, 3] *= RES
        rec = so.step(fr, bt.dt[3])
    assert [t["id"] for t in rec["tracks"]] == [int(x) for x in ta[3]["id"][:na[3]]]
    for k, t in enumerate(rec["tracks"]):
        np.testing.assert_allclose(ta[3, k]["x"], t["x"], rtol=STATE_RTOL, atol=STATE_ATOL)


def test_pose_row_scan_folded_vs_separate_kernel():
    """The pose-row scan inside pose_feature_kernel (default, S <= 4096) and pose_index_kernel (S > 4096) lay the
    rows out identically."""
    a = _run_with_env({"MMW_POSE_INDEX_FOLD": "1"})
    b = _run_with_env({"MMW_POSE_INDEX_FOLD": "0"})
    np.testing.assert_array_equal(a[1], b[1])
    np.testing.assert_array_equal(a[2], b[2])
    np.testing.assert_array_equal(a[3], b[3])
    np.testing.assert_array_equal(a[4], b[4])
    for name in ("id", "x", "P", "keypoints"):
        np.testing.assert_array_equal(a[0][name], b[0][name])


# ---- checkpoint / resume -----------------------------------------------------------------------------------
def test_dense1_wide_tiles_equal_narrow_tiles(monkeypatch):
    """Dense 1 picks 256 x 176, 256 x 192 or 256 x 256 tiles from the row count of an earlier frame (whichever needs the
    least waves-times-width on 74 CTA pairs: 72 tiles of 176 columns up to 2048 rows; 2305 rows in 192-wide tiles would
    take twice as long as 2304).  The choice must never change a bit."""
    rng = np.random.default_rng(11)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    feats = rng.normal(0, 0.4, size=(700, 3, 8, 8, 5)).astype(np.float32)
    outs = []
    for bn in ("192", "256", "176"):          # 8, 6 or 9 column tiles (the last of the 9 is 128 wide)
        monkeypatch.setenv("MMW_FC1_BN", bn)
        bt = BatchedTracker(128, max_tracks=8)
        bt.load_pose_weights(W)
        outs.append(bt.pose(feats).copy())
        bt.close()
    monkeypatch.delenv("MMW_FC1_BN")
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    assert np.abs(outs[0]).mean() > 0.05


def test_state_dump_restore_continues_bit_identically():
    S, F0, F1 = 40, 20, 12
    batches = synth.gen_batch(list(range(300, 300 + S)), F0 + F1)
    W = pw.make_pose_weights(pw.VARIANT_3D)
    a = BatchedTracker(S)
    a.load_pose_weights(W)
    for b in batches[:F0]:
        a.step(b.points, b.offsets, b.dt, pose=True)
    blob = a.state_dump()
    c = BatchedTracker(S)                       # a fresh context resumes from the blob
    c.load_pose_weights(W)
    c.state_restore(blob)
    for b in batches[F0:]:
        a.step(b.points, b.offsets, b.dt, pose=True)
        c.step(b.points, b.offsets, b.dt, pose=True)
        np.testing.assert_array_equal(a.point_assoc(), c.point_assoc())
    ta, na = a.tracks()
    tc_, nc = c.tracks()
    np.testing.assert_array_equal(na, nc)
    assert na.sum() > 40
    assert ta.tobytes() == tc_.tobytes()
    np.testing.assert_array_equal(a.ring_counts(), c.ring_counts())
    # a blob of another shape is refused
    d = BatchedTracker(S + 1)
    with pytest.raises(_lib.MmwError):
        d.state_restore(blob)


# ---- capacity limits: flagged per scene, never silent ---------------------------------------------------
def test_point_and_track_overflow_are_flagged():
    """More points in a frame than max_points_per_frame: the scene keeps the first max_points rows (and behaves
    exactly like a scene that was sent only those) and raises MMW_SCENE_POINT_OVERFLOW; more clusters than free
    track slots: MMW_SCENE_TRACK_OVERFLOW.  Other scenes of the batch are unaffected."""
    S, F, CAP = 4, 14, 96
    batches = synth.gen_batch([0, 1, 2, 3], F)
    bt = BatchedTracker(S, max_points=256)
    small = BatchedTracker(S, max_points=256)
    for b in batches:
        # scenes 1 and 3 get their frames truncated on the host for `small`, and through the device-side point
        # capacity for a context whose capacity is CAP
        bt.step(b.points, b.offsets, b.dt, pose=False)
    trunc = BatchedTracker(S, max_points=CAP)
    oracles = [mo.SceneOracle() for _ in range(S)]
    for b in batches:
        parts = [b.points[b.offsets[s]:b.offsets[s + 1]] for s in range(S)]
        # the host API refuses a batch that cannot fit the context at all ...
        cut = [p[:CAP] for p in parts]
        off = np.zeros(S + 1, np.int32)
        off[1:] = np.cumsum([len(p) for p in cut])
        small.step(np.concatenate(cut), off, b.dt, pose=False)
        recs = [o.step(cut[s], b.dt[s]) for s, o in enumerate(oracles)]
        compare_frame(small, recs, off, "truncated on the host")
    assert not small.status().any()
    # ... and the device flags scenes whose frame exceeds the per-scene capacity (device-resident input path)
    import torch
    for b in batches:
        p = torch.from_numpy(b.points).cuda()
        o = torch.from_numpy(b.offsets).cuda()
        d = torch.from_numpy(b.dt).cuda()
        trunc.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), b.points.shape[0], pose=False)
        trunc.sync()
    st = trunc.status()
    assert (st & _lib.SCENE_POINT_OVERFLOW).all()               # every scene had frames of > 96 points
    ta, na = trunc.tracks()
    tb, nb = small.tracks()
    np.testing.assert_array_equal(na, nb)                        # same as sending the first CAP rows
    for name in ("id", "x", "P"):
        np.testing.assert_array_equal(ta[name], tb[name])
    with pytest.raises(_lib.MmwError):                           # host path: more rows than S * max_points
        trunc.step(batches[0].points, batches[0].offsets, batches[0].dt, pose=False)

    # track capacity: room for 1 track, scenes with several people
    one = BatchedTracker(S, max_tracks=1)
    for b in batches:
        one.step(b.points, b.offsets, b.dt, pose=False)
    _, n1 = one.tracks()
    assert (n1 <= 1).all() and (one.status() & _lib.SCENE_TRACK_OVERFLOW).any()
    _, nfull = bt.tracks()
    assert (nfull >= n1).all() and nfull.max() > 1
