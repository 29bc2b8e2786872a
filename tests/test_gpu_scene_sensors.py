"""Per-scene sensor table and per-scene reset on the device: scenes with their own mounting, scene bound, Doppler unit
and Q format in one context, against the oracle and against contexts created with each scene's values."""
import copy

import numpy as np
import pytest

from helpers import compare_frame, oracle_config
from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, default_config
from oracle import mmw_oracle as mo

pytestmark = pytest.mark.gpu

MOUNTS = [(1.2, -15.0, 2.2), (1.8, -5.0, 2.5), (2.4, 0.0, 3.0), (1.8, 5.0, 2.5)]    # s_height, s_tilt_deg, z_max
PROFILES = [0.0626, 0.125]                                                          # m/s per Doppler bin
QFORMATS = [8, 9, 10]
S, F = 16, 60


def _params(s):
    h, t, z = MOUNTS[s % 4]
    return dict(s_height=h, s_tilt_deg=t, z_max=z, doppler_res=PROFILES[(s // 4) % 2], xyz_q_format=QFORMATS[s % 3])


def _frames(scene_ids, params, n_frames, i16=False):
    """Per frame (device rows, offsets, dt, oracle rows per scene): scene k generated as seen from its mounting, the
    Doppler column the bin index, int16 rows in the scene's Q format when i16.  The oracle gets the dequantized
    float64 values and doppler = index * unit in float64."""
    scenes = []
    for sid, p in zip(scene_ids, params):
        spec = synth.SceneSpec(s_height=p["s_height"], s_tilt_deg=p["s_tilt_deg"], doppler_res=p["doppler_res"])
        scenes.append(synth.gen_scene(sid, n_frames, spec))
    out = []
    for f in range(n_frames):
        dev, ora = [], []
        for sc, p in zip(scenes, params):
            fr = sc.frames[f]
            idx = np.rint(fr[:, 3].astype(np.float64) / p["doppler_res"])
            if i16:
                q = 2.0 ** p["xyz_q_format"]
                xyz = np.rint(fr[:, :3].astype(np.float64) * q)
                dev.append(np.concatenate([xyz, idx[:, None], fr[:, 4:5]], axis=1).astype(np.int16))
                xyz = xyz / q
            else:
                xyz = fr[:, :3].astype(np.float64)
                dev.append(np.concatenate([fr[:, :3], idx[:, None].astype(np.float32), fr[:, 4:5]], axis=1))
            ora.append(np.concatenate([xyz, (idx * p["doppler_res"])[:, None], fr[:, 4:5].astype(np.float64)], axis=1))
        off = np.zeros(len(scenes) + 1, np.int32)
        off[1:] = np.cumsum([len(d) for d in dev])
        dt = np.array([sc.dts()[f] for sc in scenes])
        out.append((np.ascontiguousarray(np.concatenate(dev, axis=0)), off, dt, ora))
    return out


def _set_table(bt, params):
    keys = ("s_height", "s_tilt_deg", "z_max", "doppler_res", "xyz_q_format")
    bt.set_scene_sensors(**{k: np.array([p[k] for p in params]) for k in keys})


def _weights():
    return pw.make_pose_weights(pw.VARIANT_3D)


@pytest.mark.parametrize("i16", [False, True], ids=["fp32", "int16"])
def test_heterogeneous_scenes_match_oracle(i16):
    params = [_params(s) for s in range(S)]
    W = _weights()
    frames = _frames(range(100, 100 + S), params, F, i16)
    bt = BatchedTracker(S)
    bt.load_pose_weights(W)
    _set_table(bt, params)
    tab = bt.scene_sensors()
    for k in ("s_height", "s_tilt_deg", "z_max", "doppler_res", "xyz_q_format"):
        np.testing.assert_array_equal(tab[k], [p[k] for p in params])
    oracles = []
    for p in params:
        cfg = oracle_config(default_config())
        cfg.s_height, cfg.s_tilt_deg, cfg.z_max = p["s_height"], p["s_tilt_deg"], p["z_max"]
        oracles.append(mo.SceneOracle(cfg, pose_weights=W))
    group = lambda s: (s % 4, (s // 4) % 2)                        # noqa: E731
    tracks, clusters = {}, {}
    for f, (pts, off, dt, ora) in enumerate(frames):
        bt.step(pts, off, dt, pose=True, record_labels=True)
        recs = [o.step(ora[s], dt[s]) for s, o in enumerate(oracles)]
        compare_frame(bt, recs, off, "frame %d" % f, labels=bt.labels(), check_keypoints=True,
                      pose_rows=bt.pose_rows())
        for s, r in enumerate(recs):
            tracks[group(s)] = tracks.get(group(s), 0) + len(r["tracks"])
            ran = r["labels"] is not None and np.any(np.asarray(r["labels"]) >= 0)
            clusters[group(s)] = clusters.get(group(s), 0) + int(ran)
    assert len(tracks) == 8 and min(tracks.values()) > 0, tracks
    assert min(clusters.values()) > 0, clusters


# ---- bitwise against contexts created with each scene's values ------------------------------------------------------
def _readback(bt, off, res=None):
    """Per scene of the last frame: every readback as bytes."""
    tr, nt = bt.tracks()
    assoc = bt.point_assoc()
    si, ti, feats = bt.pose_rows()
    rows, valid, cen = bt.export_track0()
    out = []
    for s in range(bt.S):
        sel = si == s
        d = {"tracks": tr[s].tobytes(), "n": int(nt[s]), "assoc": assoc[off[s]:off[s + 1]].tobytes(),
             "pose": (ti[sel].tobytes(), feats[sel].tobytes()), "export": (rows[s].tobytes(), bool(valid[s]),
                                                                          cen[s].tobytes())}
        if res is not None:
            d["results"] = res[s].tobytes()
        out.append(d)
    return out


def _run(bt, frames, mode, labels=False):
    """Readbacks of every frame: mode 'serial', 'pipeline' or 'run_frames' (compact records)."""
    R = bt.S * bt.tcap * _lib.RESULT_FLOATS
    out = []
    if mode == "run_frames":
        import torch
        pts = np.concatenate([fr[0] for fr in frames], axis=0)
        fro = np.cumsum([0] + [len(fr[0]) for fr in frames]).astype(np.int64)
        offs = np.stack([fr[1] for fr in frames]).astype(np.int32)
        dts = np.stack([fr[2] for fr in frames])
        res = torch.zeros(len(frames) * R, dtype=torch.float32).pin_memory().numpy().reshape(len(frames), R)
        nrec = torch.zeros(len(frames), dtype=torch.int32).pin_memory().numpy()
        bt.run_frames(pts, fro, offs, dts, res, pose=True, pipeline=True, n_records=nrec)
        full = [bt.expand_compact_results(res[f], int(nrec[f])) for f in range(len(frames))]
        return [[r.tobytes() for r in fl] for fl in full], _readback(bt, frames[-1][1])
    host = np.zeros(R, np.float32)
    for pts, off, dt, _ in frames:
        bt.step(pts, off, dt, pose=True, record_labels=labels, pipeline=mode == "pipeline")
        bt.wait_results(bt.read_results_async(host))
        d = _readback(bt, off, host.reshape(bt.S, bt.tcap, -1))
        if labels:
            lab, nf = bt.labels()
            for s in range(bt.S):
                d[s]["labels"] = (lab[s, :max(nf[s], 0)].tobytes(), int(nf[s]))
        out.append(d)
    return out


def _groups(params):
    keys = {}
    for s, p in enumerate(params):
        keys.setdefault(tuple(sorted(p.items())), []).append(s)
    return list(keys.items())


@pytest.mark.parametrize("mode", ["serial", "pipeline", "run_frames"])
def test_heterogeneous_context_equals_uniform_contexts(mode):
    params = [dict(_params(s), xyz_q_format=9) for s in range(S)]
    W = _weights()
    frames = _frames(range(200, 200 + S), params, 40)
    bt = BatchedTracker(S)
    bt.load_pose_weights(W)
    _set_table(bt, params)
    got = _run(bt, frames, mode, labels=mode == "serial")
    groups = _groups(params)
    assert len(groups) == 8
    for key, members in groups:
        p = dict(key)
        u = BatchedTracker(len(members), config=default_config(**p))
        u.load_pose_weights(W)
        sub = []
        for pts, off, dt, ora in frames:
            parts = [pts[off[s]:off[s + 1]] for s in members]
            o = np.zeros(len(members) + 1, np.int32)
            o[1:] = np.cumsum([len(x) for x in parts])
            sub.append((np.ascontiguousarray(np.concatenate(parts, axis=0)), o, dt[members], None))
        want = _run(u, sub, mode, labels=mode == "serial")
        if mode == "run_frames":
            for f in range(len(frames)):
                for k, s in enumerate(members):
                    assert got[0][f][s] == want[0][f][k], "frame %d scene %d records" % (f, s)
            got_f, want_f = [got[1]], [want[1]]
        else:
            got_f, want_f = got, want
        for f, (g, w) in enumerate(zip(got_f, want_f)):
            for k, s in enumerate(members):
                assert g[s] == w[k], "%s frame %d scene %d (%r)" % (mode, f, s, p)
        u.close()


def test_table_of_config_values_is_a_no_op():
    W = _weights()
    batches = synth.gen_batch(range(8), 30)
    frames = [(b.points, b.offsets, b.dt, None) for b in batches]
    a, b = BatchedTracker(8), BatchedTracker(8)
    cfg = a.cfg
    tab = a.scene_sensors()
    for k in ("s_height", "s_tilt_deg", "z_max", "doppler_res", "xyz_q_format"):
        assert np.all(tab[k] == getattr(cfg, k)), k
    b.set_scene_sensors(s_height=cfg.s_height, s_tilt_deg=cfg.s_tilt_deg, z_max=cfg.z_max,
                        doppler_res=cfg.doppler_res, xyz_q_format=cfg.xyz_q_format)
    for bt in (a, b):
        bt.load_pose_weights(W)
    assert _run(a, frames, "serial", labels=True) == _run(b, frames, "serial", labels=True)


def test_reset_scenes_mid_sequence_throughput_mode():
    """Scenes 2 and 5 are handed to new sensors at frame 20 (scene 5 with another mounting): they continue like fresh
    contexts of those sensors; the other scenes as if nothing had happened; frame 19's records stay valid."""
    n, F0, F1 = 8, 20, 40
    W = _weights()
    base = synth.gen_batch(range(300, 300 + n), F1)
    mount5 = dict(s_height=2.4, s_tilt_deg=0.0, z_max=3.0)
    new5 = synth.gen_scene(399, F1 - F0, synth.SceneSpec(s_height=2.4, s_tilt_deg=0.0))
    new5_dt = new5.dts()
    frames = []
    for f, b in enumerate(base):
        parts = [b.points[b.offsets[s]:b.offsets[s + 1]] for s in range(n)]
        dt = b.dt.copy()
        if f >= F0:
            parts[5] = new5.frames[f - F0]
            dt[5] = new5_dt[f - F0]
            if f == F0:
                dt[2] = 0.1
        o = np.zeros(n + 1, np.int32)
        o[1:] = np.cumsum([len(x) for x in parts])
        frames.append((np.ascontiguousarray(np.concatenate(parts, axis=0)), o, dt, None))

    def run(bt, frs, reset_at=None):
        host = np.zeros(bt.S * bt.tcap * _lib.RESULT_FLOATS, np.float32)
        out = []
        for f, (pts, off, dt, _) in enumerate(frs):
            bt.step(pts, off, dt, pose=True, pipeline=True)
            if f == reset_at:
                bt.set_scene_sensors(scenes=[5], **mount5)
                bt.reset_scenes([2, 5])
            bt.wait_results(bt.read_results_async(host))
            out.append(_readback(bt, off, host.reshape(bt.S, bt.tcap, -1)))
        return out

    a, ref = BatchedTracker(n), BatchedTracker(n)
    for bt in (a, ref):
        bt.load_pose_weights(W)
    # the reset is queued right after the step of frame F0 - 1, before that frame's records are read
    got = run(a, frames, reset_at=F0 - 1)
    want = run(ref, frames)
    for f in range(F1):
        for s in range(n):
            if s not in (2, 5) or f < F0 - 1:
                assert got[f][s] == want[f][s], "frame %d scene %d" % (f, s)
            elif f == F0 - 1:                                       # packed before the reset
                assert got[f][s]["results"] == want[f][s]["results"], "frame %d scene %d" % (f, s)
    for s, cfg in ((2, default_config()), (5, default_config(**mount5))):
        fresh = BatchedTracker(1, config=cfg)
        fresh.load_pose_weights(W)
        sub = []
        for pts, off, dt, _ in frames[F0:]:
            sub.append((np.ascontiguousarray(pts[off[s]:off[s + 1]]), np.array([0, off[s + 1] - off[s]], np.int32),
                        dt[s:s + 1], None))
        w = run(fresh, sub)
        for k in range(F1 - F0):
            assert got[F0 + k][s] == w[k][0], "frame %d scene %d after the reset" % (F0 + k, s)
        fresh.close()
    tr, nt = a.tracks()
    assert nt[2] > 0 and nt[5] > 0
    _, nid, _ = a.summary()
    _, nid_ref, _ = ref.summary()
    assert nid[2] < nid_ref[2] or nid[5] < nid_ref[5]             # ids restarted at 0


def test_set_doppler_resolution_overwrites_every_scene():
    bt = BatchedTracker(6)
    bt.set_scene_sensors(doppler_res=[0.0626, 0.125, 0.0626, 0.125, 0.25, 1.0])
    bt.set_doppler_resolution(0.0391)
    assert np.all(bt.scene_sensors()["doppler_res"] == 0.0391) and bt.cfg.doppler_res == 0.0391


def test_invalid_arguments_leave_the_table_unchanged():
    bt = BatchedTracker(4)
    bt.set_scene_sensors(s_height=[1.2, 1.8, 2.4, 3.0], doppler_res=[0.0626, 0.125, 0.0626, 0.125])
    before = bt.scene_sensors()
    lib, h = bt.lib, bt._h

    def table(**over):
        t = before.copy()
        for k, v in over.items():
            t[k][-1] = v                                            # only the last entry is bad: nothing may change
        return t

    bad = [table(s_height=np.nan), table(s_tilt_deg=np.inf), table(z_max=-np.inf), table(doppler_res=0.0),
           table(doppler_res=-0.1), table(doppler_res=np.nan), table(xyz_q_format=16), table(xyz_q_format=-1)]
    for t in bad:
        assert lib.mmw_set_scene_sensors(h, 0, 4, _lib.ptr(t)) == -1
    ok = before.copy()
    for first, n in ((-1, 1), (0, 5), (3, 2), (4, 1), (0, -1)):
        assert lib.mmw_set_scene_sensors(h, first, n, _lib.ptr(ok)) == -1, (first, n)
        assert lib.mmw_get_scene_sensors(h, first, n, _lib.ptr(ok)) == -1, (first, n)
    assert lib.mmw_set_scene_sensors(h, 0, 1, None) == -1
    assert lib.mmw_get_scene_sensors(h, 0, 1, None) == -1
    assert lib.mmw_set_doppler_resolution(h, 0.0) == -1
    for idx in ([0, 0], [4], [-1], [1, 2, 1]):
        a = np.array(idx, np.int32)
        assert lib.mmw_reset_scenes(h, _lib.ptr(a), a.size) == -1, idx
    assert lib.mmw_reset_scenes(h, None, 1) == -1
    assert bt.scene_sensors().tobytes() == before.tobytes()
    with pytest.raises(_lib.MmwError):
        bt.set_scene_sensors(doppler_res=0.0, scenes=[1])
    assert bt.scene_sensors().tobytes() == before.tobytes()


def test_preprocess_dataset_batched_mixed_radar_profiles(tmp_path, monkeypatch):
    """Three experiments logged with two radar profiles (doppler = dopplerIdx * resolution in float64, as the
    reference's reader writes it) in one run: each equals the oracle loop over its own experiment."""
    from mmwave_msc_b200 import constants, preprocessing as pp
    from mmwave_msc_b200.Utils import OfflineManager
    from test_gpu_facade import _oracle_preprocess
    monkeypatch.setattr(constants, "DOPPLER_RESOLUTION", None)
    specs = [(4, 40, 0.0626), (308, 45, 0.125), (5, 36, 0.0626)]
    dirs = []
    for sid, nf, res in specs:
        sc = synth.gen_scene(sid, nf, synth.SceneSpec(doppler_res=res))
        sc2 = copy.copy(sc)
        sc2.frames = []
        for fr in sc.frames:
            fr64 = fr.astype(np.float64)
            fr64[:, 3] = np.rint(fr64[:, 3] / res) * res                # the float64 value the reader logs
            sc2.frames.append(fr64)
        d = str(tmp_path / ("exp%d" % sid))
        synth.write_reference_csv(sc2, d, frames_per_file=20)
        dirs.append(d)
    got = pp.preprocess_dataset_batched(dirs)
    assert any(v != 0 for fr in sc2.frames for v in fr[:, 3])
    for g, d in zip(got, dirs):
        rd = OfflineManager(d)
        frames, posix, okm = [], [], []
        while not rd.is_finished():
            dok, fn, det = rd.get_data()
            okm.append(dok)
            if dok:
                frames.append(np.stack([np.asarray(det[k], np.float64) for k in
                                        ("x", "y", "z", "doppler", "peakVal")], axis=1))
                posix.append(det["posix"][0])
            else:
                frames.append(np.zeros((0, 5))); posix.append(0)
        wf, wr, wc, winv = _oracle_preprocess(frames, posix, okm, None)
        assert g.frames == wf and g.invalid_frames == winv, g.name
        for a, b in zip(g.rows, wr):
            np.testing.assert_allclose(a, b, rtol=0, atol=1e-9)
            np.testing.assert_array_equal(a[:, 3], b[:, 3])          # Doppler column: the reference's values, exactly
        for a, b in zip(g.centroids, wc):
            np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-12)
        assert len(wf) > 10


def test_checkpoint_of_heterogeneous_context_continues_bitwise():
    params = [_params(s) for s in range(S)]
    W = _weights()
    frames = _frames(range(500, 500 + S), params, 30)
    a = BatchedTracker(S)
    a.load_pose_weights(W)
    _set_table(a, params)
    _run(a, frames[:15], "serial")
    blob = a.state_dump()
    b = BatchedTracker(S)
    b.load_pose_weights(W)
    _set_table(b, params)
    b.state_restore(blob)
    assert _run(a, frames[15:], "serial") == _run(b, frames[15:], "serial")
