"""The input staging shared by the host-input entry points (mmw_step, mmw_step_packets, mmw_run_frames): one context
fed through all of them in turn gives what host mmw_step alone gives, and a refused call leaves the context as it was."""
import ctypes as C

import numpy as np
import pytest

from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, concat_packets, default_config
from oracle import tlv_oracle as tlv

pytestmark = pytest.mark.gpu

S, RES, BINS = 32, 0.0626302709636043, 256
INVALID, CAPACITY, STATE = -1, -3, -4


def _lattice(points):
    """fp32 rows on the sensor's lattice (x, y, z in Q9, Doppler column = dopplerIdx) and the same rows as int16."""
    p = points.astype(np.float64)
    q = np.stack([np.rint(p[:, 0] * 512), np.rint(p[:, 1] * 512), np.rint(p[:, 2] * 512), np.rint(p[:, 3] / RES),
                  np.rint(p[:, 4])], axis=1)
    f32 = np.stack([q[:, 0] / 512, q[:, 1] / 512, q[:, 2] / 512, q[:, 3], q[:, 4]], axis=1).astype(np.float32)
    return np.ascontiguousarray(f32), np.ascontiguousarray(q.astype(np.int16))


def _frames(seed, n_frames):
    """Per frame: fp32 rows, int16 rows, offsets, dt."""
    out = []
    for b in synth.gen_batch(list(range(seed, seed + S)), n_frames):
        f32, i16 = _lattice(b.points)
        out.append((f32, i16, b.offsets, b.dt))
    return out


def _packets(f, f32, off):
    """The frame as UART packets, and the fp32 rows mmw_step_packets decodes them into."""
    pk = [tlv.encode_packet(f + 1, f32[off[s]:off[s + 1]], 9, 1.0) for s in range(S)]
    rows = [tlv.decode_packet(p, BINS, 1.0)[2] for p in pk]
    rows = [np.zeros((0, 5)) if r is None else r for r in rows]
    ref_off = np.zeros(S + 1, np.int32)
    ref_off[1:] = np.cumsum([len(r) for r in rows])
    return pk, np.concatenate(rows).astype(np.float32), ref_off


def _tracker(W=None):
    bt = BatchedTracker(S, config=default_config(doppler_res=RES, xyz_q_format=9))
    if W is not None:
        bt.load_pose_weights(W)
    bt.set_scene_sensors(num_doppler_bins=BINS)
    return bt


def _records(bt):
    host = np.zeros(S * bt.tcap * _lib.RESULT_FLOATS, np.float32)
    bt.wait_results(bt.read_results_async(host))
    return host


# one frame per entry: (entry point, frames); run_frames groups frames by 4, so 6 frames cross a group boundary
SCHEDULE = [("f32", 1), ("i16", 1), ("packets", 1), ("run", 1), ("device", 1), ("run", 3), ("f32", 1), ("packets", 2),
            ("run", 6), ("i16", 1), ("device", 2), ("run_compact", 3), ("packets", 1), ("run", 1), ("f32", 1),
            ("i16", 1), ("run", 3)]


@pytest.mark.parametrize("pipeline", [False, True], ids=["serial", "throughput"])
def test_mixed_entry_points_on_one_context_equal_host_step(pipeline):
    import torch
    W = pw.make_pose_weights(pw.VARIANT_3D)
    F = sum(n for _, n in SCHEDULE)
    frames = _frames(1300, F)
    pk = [_packets(f, fr[0], fr[2]) for f, fr in enumerate(frames)]
    dev = [tuple(torch.from_numpy(a).cuda() for a in (fr[0], fr[2], fr[3])) for fr in frames]
    torch.cuda.synchronize()
    ref, bt = _tracker(W), _tracker(W)
    kinds = [k for k, n in SCHEDULE for _ in range(n)]
    want = []
    for f, (f32, _, off, dt) in enumerate(frames):
        if kinds[f] == "packets":
            ref.step(pk[f][1], pk[f][2], dt, pose=True)
        else:
            ref.step(f32, off, dt, pose=True)
        want.append(_records(ref))
    got = []
    f = 0
    for kind, n in SCHEDULE:
        if kind in ("f32", "i16"):
            for fr in frames[f:f + n]:
                bt.step(fr[0] if kind == "f32" else fr[1], fr[2], fr[3], pose=True, pipeline=pipeline)
                got.append(_records(bt))
        elif kind == "packets":
            for i in range(f, f + n):
                _, ok = bt.step_packets(*concat_packets(pk[i][0]), frames[i][3], pose=True, pipeline=pipeline)
                assert ok.sum() > 0
                got.append(_records(bt))
        elif kind == "device":
            for p, o, d in dev[f:f + n]:
                bt.step_device(p.data_ptr(), o.data_ptr(), d.data_ptr(), p.shape[0], pose=True, pipeline=pipeline)
                got.append(_records(bt))
        else:
            rows = [frames[i][1] for i in range(f, f + n)]     # int16 rows
            fro = np.cumsum([0] + [len(r) for r in rows]).astype(np.int64)
            offs = np.stack([frames[i][2] for i in range(f, f + n)])
            dts = np.stack([frames[i][3] for i in range(f, f + n)])
            res = torch.zeros((n, S * bt.tcap * _lib.RESULT_FLOATS), dtype=torch.float32).pin_memory().numpy()
            if kind == "run":
                bt.run_frames(np.concatenate(rows), fro, offs, dts, res, pipeline=pipeline)
                got.extend(res[i].copy() for i in range(n))
            else:
                cnt = torch.zeros(n, dtype=torch.int32).pin_memory().numpy()
                bt.run_frames(np.concatenate(rows), fro, offs, dts, res, pipeline=pipeline, n_records=cnt)
                got.extend(bt.expand_compact_results(res[i], int(cnt[i])).reshape(-1) for i in range(n))
        f += n
    assert len(got) == F
    for i in range(F):
        assert got[i].tobytes() == want[i].tobytes(), "frame %d (%s)" % (i, kinds[i])
    ta, na = ref.tracks()
    tb, nb = bt.tracks()
    assert na.sum() > S and np.array_equal(na, nb) and ta.tobytes() == tb.tobytes()
    assert bt.status().tobytes() == ref.status().tobytes()


def test_refused_calls_change_nothing():
    """Each refused mmw_step / mmw_run_frames returns its code -- the flag error first when the inputs are bad too --
    and the next valid step gives what it gives in a context that never saw the call."""
    import torch
    W = pw.make_pose_weights(pw.VARIANT_3D)
    frames = _frames(1400, 8)
    a, ref = _tracker(), _tracker(W)
    lib, h = a.lib, a._h
    n_rec = S * a.tcap * _lib.RESULT_FLOATS
    res = torch.zeros((2, n_rec), dtype=torch.float32).pin_memory().numpy()
    POSE, PIPE, I16 = _lib.STEP_POSE, _lib.STEP_PIPELINE, _lib.STEP_INPUT_I16

    def step(fr, pts=0, off=None, dt=None, flags=POSE):
        return lib.mmw_step(h, _lib.ptr(fr[0]) if pts == 0 else C.c_void_p(pts), _lib.ptr(fr[2] if off is None else off),
                            _lib.ptr(fr[3]) if dt is None else dt, flags)

    def run(fr, n=1, pts=0, fro=None, off=None, flags=POSE | PIPE | I16):
        fro = np.array([0, len(fr[1])], np.int64) if fro is None else fro
        off = np.ascontiguousarray((fr[2] if off is None else off)[None].repeat(max(n, 1), 0))
        dt = np.ascontiguousarray(fr[3][None].repeat(max(n, 1), 0))
        return lib.mmw_run_frames(h, n, _lib.ptr(fr[1]) if pts == 0 else C.c_void_p(pts), _lib.ptr(fro), _lib.ptr(off),
                                  _lib.ptr(dt), _lib.ptr(res), flags)

    assert step(frames[0]) == STATE                                 # MMW_STEP_POSE before the weights are loaded
    assert run(frames[0]) == STATE
    a.load_pose_weights(W)
    n_refused = 0
    for f, fr in enumerate(frames):
        f32, i16, off, dt = fr
        if f in (2, 5):
            bad0 = off.copy(); bad0[0] = 1
            dec = off.copy(); dec[4] = dec[5] + 1
            big = off.copy(); big[-1] = S * 256 + 1
            for flags, code in ((PIPE, STATE), (POSE | PIPE | _lib.STEP_RECORD_LABELS, INVALID)):
                assert step(fr, flags=flags) == code, flags
                assert step(fr, off=bad0, flags=flags) == code, flags
                assert run(fr, flags=flags | I16) == code, flags
                assert run(fr, off=bad0, flags=flags | I16) == code, flags
            a.set_dense_path(False)                                 # the throughput mode needs the tensor-core path
            assert step(fr, flags=POSE | PIPE) == STATE
            assert run(fr) == STATE
            a.set_dense_path(True)
            for o in (bad0, dec):
                assert step(fr, off=o) == INVALID
                assert run(fr, off=o) == INVALID
            assert step(fr, off=big) == CAPACITY
            assert run(fr, off=big) == INVALID
            assert step(fr, pts=None) == INVALID
            assert step(fr, dt=C.c_void_p(0)) == INVALID
            assert step(fr, pts=None, flags=POSE | _lib.STEP_DEVICE_INPUT) == INVALID
            assert run(fr, flags=POSE | _lib.STEP_DEVICE_INPUT) == INVALID
            assert run(fr, flags=POSE | _lib.STEP_RECORD_LABELS) == INVALID
            assert run(fr, n=-1) == INVALID
            assert run(fr, pts=None) == INVALID
            assert run(fr, fro=np.array([0, len(i16) - 1], np.int64)) == INVALID               # more points than rows
            assert run(fr, n=2, fro=np.array([0, len(i16), len(i16) - 1], np.int64)) == INVALID
            n_refused += 1
        ref.step(f32, off, dt, pose=True)
        want = _records(ref)
        if f % 2:
            a.run_frames(i16, np.array([0, len(i16)], np.int64), off[None], dt[None], res[:1])
            got = res[0]
        else:
            a.step(f32, off, dt, pose=True)
            got = _records(a)
        assert got.tobytes() == want.tobytes(), "frame %d" % f
        assert a.tracks()[0].tobytes() == ref.tracks()[0].tobytes(), "frame %d" % f
        assert a.point_assoc().tobytes() == ref.point_assoc().tobytes(), "frame %d" % f
        assert a.status().tobytes() == ref.status().tobytes(), "frame %d" % f
    assert n_refused == 2 and ref.tracks()[1].sum() > 0
