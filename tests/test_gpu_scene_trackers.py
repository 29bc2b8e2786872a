"""Per-scene tracker table on the device: scenes with their own tracker and DBSCAN constants in one context, against
the oracle and against contexts created with each scene's values; live retuning, moves, refusals and persistence."""
import numpy as np
import pytest

from helpers import compare_frame, oracle_config
from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, default_config
from oracle import mmw_oracle as mo
from oracle import tlv_oracle as tlv
from test_gpu_scene_move import _run as _run_feeds, _synth_feeds
from test_gpu_scene_sensors import _run as _run_frames

pytestmark = pytest.mark.gpu

# Four groups of settings; scene s has GROUPS[s % 4].  Group 1 is the mmw_config's defaults.
GROUPS = [
    dict(db_eps=0.2, db_min_samples=20, tr_max_tracks=2, tr_gate=4.0, tr_lifetime_dynamic=2.0, tr_lifetime_static=5.0,
         kf_q_var=0.5, kf_p_init=0.2, kf_group_disp_init=0.2, kf_spread_lim=[0.15, 0.15, 1.5, 1.0, 1.0, 0.15],
         kf_enable_est=1, x_nudge_thres=0.5, x_nudge_gain=0.3),
    dict(),
    dict(db_eps=0.45, db_min_samples=50, tr_max_tracks=10, tr_gate=6.0, tr_lifetime_dynamic=4.0, tr_lifetime_static=10.0,
         kf_q_var=2.0, kf_p_init=0.05, kf_spread_lim=[0.3, 0.3, 2.5, 1.5, 1.5, 0.3], kf_enable_est=1, kf_a_n=0.7,
         x_nudge_thres=0.8, x_nudge_gain=0.5),
    dict(db_eps=0.3, db_min_samples=20, tr_max_tracks=10, tr_gate=5.0, tr_lifetime_dynamic=1.5, tr_lifetime_static=3.0,
         kf_q_var=1.5, kf_a_spr=0.7, kf_est_pointnum=20, tr_vel_thres=0.2, x_nudge_thres=1.0, x_nudge_gain=0.4),
]
TCAP = 16                 # above every group's tr_max_tracks: no capacity overflow where the oracle has none
FIELDS = _lib.SCENE_TRACKER_DTYPE.names


def _weights():
    return pw.make_pose_weights(pw.VARIANT_3D)


def _set_entries(bt, entries, scenes=None):
    """Sets each listed scene's entry: the mmw_config's values overridden by entries[k]."""
    idx = list(range(bt.S)) if scenes is None else list(scenes)
    full = [default_config(**e) for e in entries]
    bt.set_scene_trackers(scenes=idx, **{k: np.array([(list(getattr(c, k)) if k == "kf_spread_lim" else getattr(c, k))
                                                      for c in full]) for k in FIELDS})


def _oracle_cfg(entry):
    c = default_config(**entry)
    o = oracle_config(c)
    o.x_nudge_thres, o.x_nudge_gain = c.x_nudge_thres, c.x_nudge_gain
    return o


def _retune(oracle, cfg):
    """The oracle scene continues under cfg: the scene's and every live track's constants replaced."""
    oracle.cfg = cfg
    for t in oracle.tracks:
        t.cfg = cfg


def _ran_dbscan(rec):
    return rec["labels"] is not None and bool(np.any(np.asarray(rec["labels"]) >= 0))


# ---- 1: a heterogeneous fleet against the oracle ------------------------------------------------------------------
def test_heterogeneous_fleet_matches_oracle():
    S, F = 16, 60
    W = _weights()
    batches = synth.gen_batch(range(700, 700 + S), F)
    bt = BatchedTracker(S, max_tracks=TCAP)
    bt.load_pose_weights(W)
    entries = [GROUPS[s % 4] for s in range(S)]
    _set_entries(bt, entries)
    tab = bt.scene_trackers()
    for s, e in enumerate(entries):
        for k, v in e.items():
            np.testing.assert_array_equal(tab[k][s], v, err_msg=k)
    oracles = [mo.SceneOracle(_oracle_cfg(e), pose_weights=W) for e in entries]
    tracks, clusters = [0] * 4, [0] * 4
    for f, b in enumerate(batches):
        bt.step(b.points, b.offsets, b.dt, pose=True, record_labels=True)
        recs = [o.step(b.points[b.offsets[s]:b.offsets[s + 1]], b.dt[s]) for s, o in enumerate(oracles)]
        compare_frame(bt, recs, b.offsets, "frame %d" % f, labels=bt.labels(), check_keypoints=True,
                      pose_rows=bt.pose_rows())
        for s, r in enumerate(recs):
            tracks[s % 4] += len(r["tracks"])
            clusters[s % 4] += int(_ran_dbscan(r))
    assert min(tracks) > 0 and min(clusters) > 0, (tracks, clusters)


# ---- 2: bitwise against one context per scene ---------------------------------------------------------------------
PROFILE = dict(num_doppler_bins=32, doppler_res=0.0626, xyz_q_format=9)


def _packet_feeds(seed, S, F):
    out = []
    for s in range(S):
        sc = synth.gen_scene(seed + s, F, synth.SceneSpec(doppler_res=PROFILE["doppler_res"]))
        out.append([(tlv.encode_packet(f + 1, sc.frames[f], PROFILE["xyz_q_format"], PROFILE["doppler_res"]),
                     float(sc.dts()[f])) for f in range(F)])
    return out


def _frames_of(feeds):
    """feeds[s][f] -> frames in the layout test_gpu_scene_sensors._run takes."""
    out = []
    for f in range(len(feeds[0])):
        rows = [fd[f][0] for fd in feeds]
        off = np.zeros(len(feeds) + 1, np.int32)
        off[1:] = np.cumsum([len(r) for r in rows])
        out.append((np.ascontiguousarray(np.concatenate(rows, axis=0)), off,
                    np.array([fd[f][1] for fd in feeds], np.float64), None))
    return out


def _ctx(S, W, cfg=None, packets=False):
    bt = BatchedTracker(S, max_tracks=TCAP, config=cfg)
    bt.load_pose_weights(W)
    if packets:
        bt.set_scene_sensors(**PROFILE)
    return bt


@pytest.mark.parametrize("mode", ["serial", "pipeline", "run_frames", "packets"])
def test_heterogeneous_context_equals_one_context_per_scene(mode):
    S, F = 8, 30
    W = _weights()
    packets = mode == "packets"
    feeds = _packet_feeds(800, S, F) if packets else _synth_feeds(800, S, F)
    entries = [GROUPS[s % 4] for s in range(S)]
    het = _ctx(S, W, packets=packets)
    _set_entries(het, entries)

    def run(bt, fds):
        if mode == "run_frames":
            return _run_frames(bt, _frames_of(fds), "run_frames")
        return _run_feeds(bt, fds, range(F), pipeline=mode == "pipeline", packets=packets)

    got = run(het, feeds)
    for s in range(S):
        one = _ctx(1, W, default_config(**entries[s]), packets=packets)
        want = run(one, [feeds[s]])
        if mode == "run_frames":
            for f in range(F):
                assert got[0][f][s] == want[0][f][0], "frame %d scene %d records" % (f, s)
            assert got[1][s] == want[1][0], "scene %d readback" % s
        else:
            for f in range(F):
                assert got[f][s] == want[f][0], "%s frame %d scene %d" % (mode, f, s)
        one.close()


# ---- 3: live retune -----------------------------------------------------------------------------------------------
K = 15                    # the entries change between frame K - 1 and frame K


def _state_hist(bt, blob):
    """(S, 3, 272) ring histograms out of a state blob (mmw_state_dump layout: header, then the parts in order)."""
    S, n, t = bt.S, bt.ncap, bt.tcap
    o = 32 + 64 * S + 1264 * S * t + 4 * S * t * 3 * 64 * 5 + 4 * S * 3 * n * 5
    assert blob.size == o + 272 * 3 * S + 4 * S * t * 57 + 4 * S == bt.lib.mmw_state_size(bt._h)
    return blob[o:o + 272 * 3 * S].reshape(S, 3, 272)


def _flags(bt):
    return _state_hist(bt, bt.state_dump())[:, :, 256:260].copy().view(np.uint32)[:, :, 0]


def _eps_raise_scene(F):
    """A scene that is empty until frame K - 2, then holds 17 points at x = -1.2 (frame K - 2), 17 at x = +1.2 (K - 1)
    and one at x = 0 (K), all at y' = 2, z' = 1.  Under db_eps = 1.5 the middle point reaches both groups: 35 points,
    one core point, one cluster at frame K.  The groups were binned under db_eps = 0.3 (cells 0.69 m wide: x = -1.2,
    0 and 1.2 fall in cells 6, 8 and 9), so the summed histogram holds at most 18 points around any cell."""
    frames = [np.zeros((0, 5), np.float32) for _ in range(F)]
    j = (np.arange(17) - 8) / 800.0
    frames[K - 2] = synth.raw_from_world(-1.2 + j, np.full(17, 2.0), np.ones(17), np.zeros(17), np.full(17, 100.0))
    frames[K - 1] = synth.raw_from_world(1.2 + j, np.full(17, 2.0), np.ones(17), np.zeros(17), np.full(17, 100.0))
    frames[K] = synth.raw_from_world([0.0], [2.0], [1.0], [0.0], [100.0])
    return frames


def test_live_retune_continues_every_scene_under_its_new_constants():
    S, F = 8, 40
    W = _weights()
    feeds = _synth_feeds(900, S, F)
    raise_frames = _eps_raise_scene(F)
    feeds[0] = [(raise_frames[f], 0.1) for f in range(F)]
    new = {0: dict(db_eps=1.5),                                              # DBSCAN: the cluster of frame K
           1: dict(tr_gate=6.0, tr_lifetime_dynamic=1.5, kf_q_var=2.0),      # tracker only: flags stay as they are
           2: dict(db_min_samples=20, tr_max_tracks=2),
           3: GROUPS[2],
           5: dict(kf_p_init=0.3, kf_group_disp_init=0.05, kf_spread_lim=[0.3] * 6, kf_enable_est=1)}
    bt = BatchedTracker(S, max_tracks=TCAP)
    bt.load_pose_weights(W)
    oracles = [mo.SceneOracle(_oracle_cfg({}), pose_weights=W) for _ in range(S)]
    frames = _frames_of(feeds)
    spawned_at_k = None
    for f, (pts, off, dt, _) in enumerate(frames):
        if f == K:
            before = _flags(bt)
            _set_entries(bt, [new[s] for s in sorted(new)], scenes=sorted(new))
            after = _flags(bt)
            for s, e in new.items():
                _retune(oracles[s], _oracle_cfg(e))
        bt.step(pts, off, dt, pose=True, record_labels=True)
        recs = [o.step(pts[off[s]:off[s + 1]].astype(np.float64), dt[s]) for s, o in enumerate(oracles)]
        compare_frame(bt, recs, off, "frame %d" % f, labels=bt.labels(), check_keypoints=True,
                      pose_rows=bt.pose_rows())
        if f == K:
            spawned_at_k = len(recs[0]["tracks"])
    assert spawned_at_k == 1
    assert bt.scene_trackers()["db_eps"][0] == 1.5
    # (checked after the frames, so that a missing flag shows first as the missed cluster of frame K)
    for s in range(S):
        if s in (0, 2, 3):                                   # a DBSCAN field changed: every ring histogram flagged
            assert np.all(after[s] == 1), (s, after[s])
        else:                                                # tracker fields only, or no change: flags as they were
            assert np.array_equal(after[s], before[s]), s


# ---- 4: identity --------------------------------------------------------------------------------------------------
def test_table_of_config_values_is_a_no_op():
    W = _weights()
    frames = _frames_of(_synth_feeds(950, 8, 30))
    a, b = BatchedTracker(8), BatchedTracker(8)
    tab = a.scene_trackers()
    for k in FIELDS:
        v = getattr(a.cfg, k)
        assert np.all(tab[k] == (list(v) if k == "kf_spread_lim" else v)), k
    _set_entries(b, [{}] * 8)
    assert b.scene_trackers().tobytes() == tab.tobytes()
    for bt in (a, b):
        bt.load_pose_weights(W)
    b.state_restore(a.state_dump())       # the same bytes everywhere, the rings' never-written rows included
    assert _run_frames(a, frames[:15], "serial", labels=True) == _run_frames(b, frames[:15], "serial", labels=True)
    assert a.state_dump().tobytes() == b.state_dump().tobytes()
    _set_entries(b, [{}] * 8)                                               # also on live scenes
    assert a.state_dump().tobytes() == b.state_dump().tobytes()
    assert _run_frames(a, frames[15:], "serial", labels=True) == _run_frames(b, frames[15:], "serial", labels=True)
    assert a.state_dump().tobytes() == b.state_dump().tobytes()


# ---- 5: moves -----------------------------------------------------------------------------------------------------
def test_move_with_and_without_the_entry():
    S, F0, F = 4, 20, 40
    W = _weights()
    feeds = _synth_feeds(960, S, F)
    tuned = GROUPS[2]
    # the destination's defaults differ from the tuned entry in every tracker field, not in the DBSCAN ones (the ring
    # histograms travel as they are: see mmw_import_scenes)
    dest = dict(tr_max_tracks=3, tr_gate=5.5, tr_lifetime_dynamic=2.5, tr_lifetime_static=6.0, kf_q_var=0.8,
                kf_p_init=0.15, kf_spread_lim=[0.25] * 6, x_nudge_gain=0.2,
                **{k: tuned[k] for k in ("db_eps", "db_min_samples")})
    a = _ctx(S, W)
    _set_entries(a, [tuned], scenes=[1])
    src_entry = a.scene_trackers()[1:2].copy()
    blob = {}
    got_a = _run_feeds(a, feeds, range(F), hooks={F0 - 1: lambda: blob.update(b=a.export_scenes([1]))})
    # with the entry: slot 2 of b continues as scene 1 of a
    b = _ctx(S, W, default_config(**dest))
    _run_feeds(b, feeds, range(F0))
    b.import_scenes(blob["b"], [2])
    assert b.lib.mmw_set_scene_trackers(b._h, 2, 1, _lib.ptr(src_entry)) == 0
    moved = [list(fd) for fd in feeds]
    moved[2] = feeds[1]
    got_b = _run_feeds(b, moved, range(F0, F))
    for f in range(F0, F):
        assert got_b[f - F0][2] == got_a[f][1], "frame %d" % f
    # without it: slot 2 of c runs under c's entry, which the oracle confirms
    c = _ctx(S, W, default_config(**dest))
    oracles = [mo.SceneOracle(_oracle_cfg(dest), pose_weights=W) for _ in range(S)]
    oracles[2] = mo.SceneOracle(_oracle_cfg(tuned), pose_weights=W)      # scene 1 of a, up to the move
    frames = _frames_of(feeds)
    for f in range(F0):
        pts, off, dt, _ = frames[f]
        c.step(pts, off, dt, pose=True)
        for s, o in enumerate(oracles):
            src = 1 if s == 2 else s
            o.step(pts[off[src]:off[src + 1]].astype(np.float64), dt[src])
    c.import_scenes(blob["b"], [2])
    assert c.scene_trackers()[2]["tr_max_tracks"] == 3
    _retune(oracles[2], _oracle_cfg(dest))
    frames = _frames_of(moved)
    for f in range(F0, F):
        pts, off, dt, _ = frames[f]
        c.step(pts, off, dt, pose=True, record_labels=True)
        recs = [o.step(pts[off[s]:off[s + 1]].astype(np.float64), dt[s]) for s, o in enumerate(oracles)]
        compare_frame(c, recs, off, "frame %d" % f, labels=c.labels(), check_keypoints=True, pose_rows=c.pose_rows())


# ---- 6: refusals and persistence ----------------------------------------------------------------------------------
def test_invalid_entries_change_nothing_and_queue_nothing():
    W = _weights()
    bt = BatchedTracker(4)
    bt.load_pose_weights(W)
    _run_frames(bt, _frames_of(_synth_feeds(970, 4, 6)), "serial")
    _set_entries(bt, [GROUPS[0], {}, GROUPS[2], GROUPS[3]])
    before = bt.scene_trackers()
    state = bt.state_dump().tobytes()
    lib, h = bt.lib, bt._h

    def table(field, value, k=None):
        t = before.copy()
        t["db_eps"][0] = 0.9                                   # a change that would raise scene 0's flags if queued
        if k is None:
            t[field][-1] = value                               # only the last entry is bad
        else:
            t[field][-1, k] = value
        return t

    bad = []
    for name in FIELDS:
        if _lib.SCENE_TRACKER_DTYPE[name].kind == "f" or _lib.SCENE_TRACKER_DTYPE[name].base.kind == "f":
            for v in (np.nan, np.inf, -np.inf):
                if name == "kf_spread_lim":
                    bad += [table(name, v, k) for k in range(6)]
                else:
                    bad.append(table(name, v))
    bad += [table("db_min_samples", 0), table("db_min_samples", -3), table("tr_max_tracks", -1)]
    for t in bad:
        assert lib.mmw_set_scene_trackers(h, 0, 4, _lib.ptr(t)) == -1
    ok = before.copy()
    for first, n in ((-1, 1), (0, 5), (3, 2), (4, 1), (0, -1)):
        assert lib.mmw_set_scene_trackers(h, first, n, _lib.ptr(ok)) == -1, (first, n)
        assert lib.mmw_get_scene_trackers(h, first, n, _lib.ptr(ok)) == -1, (first, n)
    assert lib.mmw_set_scene_trackers(h, 0, 1, None) == -1
    assert lib.mmw_get_scene_trackers(h, 0, 1, None) == -1
    assert lib.mmw_set_scene_trackers(None, 0, 1, _lib.ptr(ok)) == -1
    assert bt.scene_trackers().tobytes() == before.tobytes()
    assert bt.state_dump().tobytes() == state
    with pytest.raises(_lib.MmwError):
        bt.set_scene_trackers(db_min_samples=0, scenes=[1])
    assert bt.scene_trackers().tobytes() == before.tobytes()
    assert bt.state_dump().tobytes() == state
    # the edge values mmw_create accepts are accepted here too
    _set_entries(bt, [dict(db_min_samples=1, tr_max_tracks=0)], scenes=[3])
    assert bt.scene_trackers()[3]["tr_max_tracks"] == 0


def test_table_survives_resets_restore_and_import():
    W = _weights()
    bt = _ctx(4, W)
    _set_entries(bt, [GROUPS[0], GROUPS[2], {}, GROUPS[3]])
    want = bt.scene_trackers().tobytes()
    feeds = _synth_feeds(980, 4, 8)
    _run_feeds(bt, feeds, range(8))
    blob = bt.state_dump()
    sblob = bt.export_scenes([0, 1])
    bt.reset()
    assert bt.scene_trackers().tobytes() == want
    bt.reset_scenes([1, 3])
    assert bt.scene_trackers().tobytes() == want
    bt.state_restore(blob)
    assert bt.scene_trackers().tobytes() == want
    bt.import_scenes(sblob, [2, 3])
    assert bt.scene_trackers().tobytes() == want
    other = _ctx(4, W, default_config(tr_max_tracks=7))
    other.import_scenes(sblob, [0, 1])
    assert np.all(other.scene_trackers()["tr_max_tracks"] == 7)
