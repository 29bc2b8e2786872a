"""Stepping a fleet straight from its sensors' UART packets (mmw_step_packets): scenes with three radar profiles (own
numDopplerBins, Doppler resolution and Q format) in one context, against the reference decoder + oracle, against
mmw_decode_tlv + mmw_step, in throughput mode, and after refused calls."""
import ctypes as C

import numpy as np
import pytest

from helpers import compare_frame
from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, concat_packets
from oracle import mmw_oracle as mo
from oracle import tlv_oracle as tlv

pytestmark = pytest.mark.gpu

PROFILES = [(16, 0.125, 8), (32, 0.0626, 9), (64, 0.0391, 10)]     # numDopplerBins, dopplerResolutionMps, xyzQFormat
S, F, NCAP = 12, 40, 300
NO_PACKET, BAD, OVER = 9, 10, 11                                   # scenes with gaps, dataOK = 0 frames, > NCAP objects


def _profile(s):
    return PROFILES[s % 3]


def _fleet(seed, n_frames=F):
    """Per frame: (packets [S] (bytes or None), dt [S]).  Scene OVER sends two people's scenes in one packet."""
    scenes, dts = [], []
    for s in range(S):
        res = _profile(s)[1]
        sc = synth.gen_scene(seed + s, n_frames, synth.SceneSpec(doppler_res=res))
        scenes.append(sc)
        dts.append(sc.dts())
    extra = synth.gen_scene(seed + 99, n_frames, synth.SceneSpec(doppler_res=_profile(OVER)[1]))
    out = []
    for f in range(n_frames):
        pk = []
        for s in range(S):
            bins, res, q = _profile(s)
            rows = scenes[s].frames[f]
            if s == OVER:
                rows = np.concatenate([rows, extra.frames[f]], axis=0)
            p = tlv.encode_packet(f + 1, rows, q, res)
            if s == NO_PACKET and f % 4 == 1:
                p = None
            elif s == BAD and f % 3 == 2:
                kind = (f // 3) % 4
                p = [tlv.encode_packet(f + 1, rows, q, res, tlv_type=2), p[:-5], b"\x09" + p[1:],
                     tlv.encode_packet(f + 1, np.zeros((0, 5)), q, res)][kind]
            pk.append(p)
        out.append((pk, np.array([d[f] for d in dts])))
    return out


def _tracker(W, table=True):
    bt = BatchedTracker(S, max_points=NCAP)
    bt.load_pose_weights(W)
    if table:
        bt.set_scene_sensors(doppler_res=[_profile(s)[1] for s in range(S)],
                             num_doppler_bins=[_profile(s)[0] for s in range(S)])
    return bt


def _readback(bt, host=None):
    tr, nt = bt.tracks()
    lab, nf = bt.labels()                                            # only the first n_fused labels of a scene are defined
    d = {"tracks": tr.tobytes(), "n": nt.tobytes(), "status": bt.status().tobytes(),
         "assoc": bt.point_assoc().tobytes(), "labels": [(lab[s, :max(nf[s], 0)].tobytes(), int(nf[s]))
                                                         for s in range(bt.S)]}
    if host is not None:
        d["results"] = host.tobytes()
    return d


def test_mixed_fleet_matches_reference_decoder_and_oracle():
    W = pw.make_pose_weights(pw.VARIANT_3D)
    bt = _tracker(W)
    oracles = [mo.SceneOracle(pose_weights=W) for _ in range(S)]
    n_tracks = np.zeros(S, np.int64)
    kinds = set()
    for f, (pk, dt) in enumerate(_fleet(700)):
        blob, off = concat_packets(pk)
        frames, ok = bt.step_packets(blob, off, dt, pose=True, record_labels=True)
        rows, recs = [], []
        for s, p in enumerate(pk):
            bins, res, _ = _profile(s)
            wok, wframe, r = tlv.decode_packet(p, bins, res) if p is not None else (0, 0, None)
            assert (bool(ok[s]), int(frames[s])) == (bool(wok), wframe), "frame %d scene %d" % (f, s)
            r = r if wok else np.zeros((0, 5))
            rows.append(len(r))
            kinds.add((s, "none" if p is None else ("bad" if not wok else ("over" if len(r) > NCAP else "ok"))))
            recs.append(oracles[s].step(r[:NCAP], dt[s]))
        off_rows = np.zeros(S + 1, np.int64)
        off_rows[1:] = np.cumsum(rows)
        off_rows[S] = off_rows[S - 1] + min(rows[S - 1], NCAP)      # the device keeps the first NCAP rows of OVER
        compare_frame(bt, recs, off_rows, "frame %d" % f, labels=bt.labels(), check_keypoints=True,
                      pose_rows=bt.pose_rows())
        n_tracks += [len(r["tracks"]) for r in recs]
    assert (NO_PACKET, "none") in kinds and (BAD, "bad") in kinds and (OVER, "over") in kinds
    st = bt.status()
    assert st[OVER] & _lib.SCENE_POINT_OVERFLOW and not (st[:OVER] & _lib.SCENE_POINT_OVERFLOW).any()
    for g in range(3):                                              # every profile tracked people
        assert n_tracks[g::3].sum() > 0, g


def _run_packets(bt, fleet, pipeline=False, labels=True):
    host = np.zeros(S * bt.tcap * _lib.RESULT_FLOATS, np.float32)
    out = []
    for pk, dt in fleet:
        blob, off = concat_packets(pk)
        bt.step_packets(blob, off, dt, pose=True, record_labels=labels, pipeline=pipeline)
        bt.wait_results(bt.read_results_async(host))
        out.append(_readback(bt, host))
    return out


def test_equals_decode_tlv_then_step():
    """Per-profile mmw_decode_tlv (in the context's unit 1.0: rows carry dopplerIdx) + mmw_step on the same table."""
    W = pw.make_pose_weights(pw.VARIANT_3D)
    fleet = _fleet(800)
    got = _run_packets(_tracker(W), fleet)
    ref = _tracker(W, table=False)
    ref.set_scene_sensors(doppler_res=[_profile(s)[1] for s in range(S)])
    host = np.zeros(S * ref.tcap * _lib.RESULT_FLOATS, np.float32)
    launches = []
    for f, (pk, dt) in enumerate(fleet):
        parts = [None] * S
        for g, (bins, _, _) in enumerate(PROFILES):
            members = list(range(g, S, 3))
            pts, poff, _, _ = ref.decode_tlv([pk[s] or b"" for s in members], bins, 1.0)
            for k, s in enumerate(members):
                parts[s] = pts[poff[k]:poff[k + 1]]
        off = np.zeros(S + 1, np.int32)
        off[1:] = np.cumsum([len(p) for p in parts])
        ref.step(np.concatenate(parts, axis=0), off, dt, pose=True, record_labels=True)
        ref.wait_results(ref.read_results_async(host))
        assert _readback(ref, host) == got[f], "frame %d" % f
    assert any(np.frombuffer(g["n"], np.int32).sum() > 0 for g in got)


def test_throughput_mode_equals_serial():
    W = pw.make_pose_weights(pw.VARIANT_3D)
    fleet = _fleet(900)
    serial = _run_packets(_tracker(W), fleet, labels=False)
    bt = _tracker(W)
    piped = _run_packets(bt, fleet, pipeline=True, labels=False)
    for f, (a, b) in enumerate(zip(serial, piped)):
        for k in ("tracks", "n", "status", "assoc", "results"):
            assert a[k] == b[k], "frame %d %s" % (f, k)
    prof = bt.profile_kernels(lambda i: bt.step_packets(*concat_packets(fleet[i][0]), fleet[i][1], pipeline=True), 3)
    assert prof.get("packets", 0.0) > 0.0, prof


def test_refused_calls_change_nothing():
    """Each refused call returns its code before anything is queued: the next valid step gives what it gives in a
    context that never saw the call, and frame_numbers / data_ok are left alone."""
    W = pw.make_pose_weights(pw.VARIANT_3D)
    fleet = _fleet(1000, 12)
    a, ref = _tracker(W, table=False), _tracker(W)
    lib, h = a.lib, a._h
    fr = np.full(S, -7, np.int32)
    ok = np.full(S, -7, np.int32)

    def call(blob, off, dt, flags=_lib.STEP_POSE | _lib.STEP_RECORD_LABELS, blob_p=None, off_p=None, dt_p=None):
        return lib.mmw_step_packets(h, blob_p if blob_p is not None else _lib.ptr(blob),
                                    off_p if off_p is not None else _lib.ptr(off),
                                    dt_p if dt_p is not None else _lib.ptr(dt), flags, _lib.ptr(fr), _lib.ptr(ok))

    blob, off = concat_packets(fleet[0][0])
    assert call(blob, off, fleet[0][1]) == -4                       # MMW_ERR_STATE: no num_doppler_bins in the table yet
    a.set_scene_sensors(doppler_res=[_profile(s)[1] for s in range(S)],
                        num_doppler_bins=[_profile(s)[0] for s in range(S)])
    n_refused = 0
    for f, (pk, dt) in enumerate(fleet):
        blob, off = concat_packets(pk)
        if f in (3, 7):
            big = list(pk)
            big[2] = tlv.encode_packet(1, np.zeros((S * NCAP + 1, 5)), 9, 0.0626)
            assert call(*concat_packets(big), dt) == -3                              # MMW_ERR_CAPACITY
            bad0 = off.copy(); bad0[0] = 1
            dec = off.copy(); dec[4] = dec[5] + 1
            past = off.copy(); past[-1] = -1
            for o in (bad0, dec, past):
                assert call(blob, o, dt) == -1, o                                    # MMW_ERR_INVALID
            assert call(blob, off, dt, dt_p=C.c_void_p(0)) == -1
            assert call(blob, off, dt, off_p=C.c_void_p(0)) == -1
            assert call(blob, off, dt, blob_p=C.c_void_p(0)) == -1
            for flags in (_lib.STEP_POSE | _lib.STEP_INPUT_I16, _lib.STEP_POSE | _lib.STEP_DEVICE_INPUT,
                          _lib.STEP_POSE | _lib.STEP_PIPELINE | _lib.STEP_RECORD_LABELS):
                assert call(blob, off, dt, flags=flags) == -1, flags
            a.set_scene_sensors(num_doppler_bins=0, scenes=[5])
            assert call(blob, off, dt) == -4                                         # MMW_ERR_STATE
            a.set_scene_sensors(num_doppler_bins=_profile(5)[0], scenes=[5])
            assert (fr == -7).all() and (ok == -7).all()
            n_refused += 1
        assert call(blob, off, dt) == 0
        ref.step_packets(blob, off, dt, pose=True, record_labels=True)
        a._n_last = ref._n_last
        assert _readback(a) == _readback(ref), "frame %d" % f
        np.testing.assert_array_equal(ok.astype(bool), [p is not None and tlv.decode_packet(p, 16, 1.0)[0] == 1
                                                        for p in pk])
        fr[:] = -7
        ok[:] = -7
    assert n_refused == 2


def test_num_doppler_bins_round_trips_and_negative_changes_nothing():
    bt = BatchedTracker(4)
    assert (bt.scene_sensors()["num_doppler_bins"] == 0).all()      # mmw_create: not set
    bt.set_scene_sensors(num_doppler_bins=[16, 32, 64, 0], doppler_res=[0.125, 0.0626, 0.0391, 1.0])
    tab = bt.scene_sensors()
    np.testing.assert_array_equal(tab["num_doppler_bins"], [16, 32, 64, 0])
    np.testing.assert_array_equal(tab["doppler_res"], [0.125, 0.0626, 0.0391, 1.0])
    bt.set_scene_sensors(s_height=2.0)                              # other fields leave it alone
    np.testing.assert_array_equal(bt.scene_sensors()["num_doppler_bins"], [16, 32, 64, 0])
    before = bt.scene_sensors()
    t = before.copy()
    t["num_doppler_bins"][-1] = -1
    assert bt.lib.mmw_set_scene_sensors(bt._h, 0, 4, _lib.ptr(t)) == -1
    with pytest.raises(_lib.MmwError):
        bt.set_scene_sensors(num_doppler_bins=-16, scenes=[1])
    assert bt.scene_sensors().tobytes() == before.tobytes()
    bt.set_doppler_resolution(0.5)                                   # sets every unit, keeps the bins
    np.testing.assert_array_equal(bt.scene_sensors()["num_doppler_bins"], [16, 32, 64, 0])
