"""Per-scene export and import of tracker state: live scenes moved between contexts, slots and GPUs continue bit for
bit as if they had never moved, and a malformed scene blob changes nothing."""
import numpy as np
import pytest

from mmwave_msc_b200 import _lib, pose_weights as pw, synth
from mmwave_msc_b200.batched import BatchedTracker, concat_packets, scene_blob_info
from mmwave_msc_b200.sharding import move_scenes
from oracle import tlv_oracle as tlv
from test_gpu_scene_sensors import _frames, _params

pytestmark = pytest.mark.gpu


def _weights():
    return pw.make_pose_weights(pw.VARIANT_3D)


def _tracker(S, W, device=0, max_points=256, max_tracks=8):
    bt = BatchedTracker(S, max_points=max_points, max_tracks=max_tracks, device=device)
    bt.load_pose_weights(W)
    return bt


def _synth_feeds(seed, S, F):
    """feeds[s][f] = (rows (N, 5) float32, dt) of synthetic scene seed + s."""
    out = []
    for s in range(S):
        sc = synth.gen_scene(seed + s, F)
        out.append([(sc.frames[f], float(sc.dts()[f])) for f in range(F)])
    return out


def _feeds_from_frames(frames):
    """feeds in the layout of test_gpu_scene_sensors._frames (device rows, offsets, dt, oracle rows)."""
    S = len(frames[0][2])
    return [[(fr[0][fr[1][s]:fr[1][s + 1]], float(fr[2][s])) for fr in frames] for s in range(S)]


def _after(feeds, f0, moves):
    """Inputs of a context whose slot d takes over the feed of scene s from frame f0 on, for (s, d, src) in moves
    (src: the feeds the scene came from)."""
    out = [list(fd) for fd in feeds]
    for s, d, src in moves:
        out[d][f0:] = src[s][f0:]
    return out


def _step(bt, items, pipeline, labels, packets):
    dt = np.array([it[1] for it in items], np.float64)
    if packets:
        blob, off = concat_packets([it[0] for it in items])
        _, ok = bt.step_packets(blob, off, dt, pose=True, record_labels=labels, pipeline=pipeline)
        rows = [int.from_bytes(it[0][44:46], "little") if k else 0 for it, k in zip(items, ok)]
    else:
        rows_l = [it[0] for it in items]
        pts = np.ascontiguousarray(np.concatenate(rows_l, axis=0))
        rows = [len(r) for r in rows_l]
        off = np.zeros(len(items) + 1, np.int32)
        off[1:] = np.cumsum(rows)
        bt.step(pts, off, dt, pose=True, record_labels=labels, pipeline=pipeline)
    off = np.zeros(len(items) + 1, np.int64)
    off[1:] = np.cumsum(rows)
    return off


def _views(bt, off, host, labels):
    """Everything readable about each scene after a frame, as bytes."""
    tr, nt = bt.tracks()
    n, nid, lm = bt.summary()
    rc = bt.ring_counts()
    st = bt.status()
    assoc = bt.point_assoc()
    lab, nf = bt.labels() if labels else (None, None)
    rec = host.reshape(bt.S, bt.tcap, -1)
    out = []
    for s in range(bt.S):
        d = {"tracks": tr[s].tobytes(), "summary": (int(nt[s]), int(nid[s]), int(lm[s])), "ring": rc[s].tobytes(),
             "status": int(st[s]), "results": rec[s].tobytes(), "assoc": assoc[off[s]:off[s + 1]].tobytes()}
        if labels:
            d["labels"] = (lab[s, :max(nf[s], 0)].tobytes(), int(nf[s]))
        out.append(d)
    return out


def _run(bt, feeds, f_range, pipeline=False, hooks=None, packets=False, views=True):
    """Steps frames f_range of the per-slot feeds; hooks[f]() runs right after frame f's step, before its records
    are read.  Returns the views of every frame."""
    labels = not pipeline
    host = np.zeros(bt.S * bt.tcap * _lib.RESULT_FLOATS, np.float32)
    out = []
    for f in f_range:
        off = _step(bt, [fd[f] for fd in feeds], pipeline, labels, packets)
        if hooks and f in hooks:
            hooks[f]()
        bt.wait_results(bt.read_results_async(host))
        out.append(_views(bt, off, host, labels) if views else None)
    return out


STATE_KEYS = ("tracks", "summary", "ring", "status", "results")     # what an import carries into the records at once


def _same_scene(got, want, ctx, keys=None):
    for k in keys or want:
        assert got[k] == want[k], "%s: %s differs" % (ctx, k)


# ---- 1, 2, 7: move mid-sequence ---------------------------------------------------------------------------------
S1, F0, F1 = 16, 20, 25
MOVES = ((3, 0), (7, 9), (11, 4))                                    # scene of A -> slot of B


def _device_records(bt):
    import torch
    buf = torch.zeros(bt.S * bt.tcap * _lib.RESULT_FLOATS, dtype=torch.float32, device=torch.device("cuda", bt.device))
    bt.pack_results(buf.data_ptr())
    bt.sync()
    return buf.cpu().numpy().reshape(bt.S, -1)


def _move_mid_sequence(pipeline, device_b=0):
    W = _weights()
    fa, fb = _synth_feeds(0, S1, F0 + F1), _synth_feeds(100, S1, F0 + F1)
    a, b, r = _tracker(S1, W), _tracker(S1, W, device=device_b), _tracker(S1, W, device=device_b)
    src = [s for s, _ in MOVES]
    dst = [d for _, d in MOVES]
    fb_after = _after(fb, F0, [(s, d, fa) for s, d in MOVES])
    packed = {}

    def export():
        packed["blob"] = a.export_scenes(src)
        if not pipeline:
            packed["a"] = _device_records(a)

    def imp():
        b.import_scenes(packed["blob"], dst)
        if not pipeline:
            packed["b"] = _device_records(b)

    got_a = _run(a, fa, range(F0 + F1), pipeline, hooks={F0 - 1: export})
    got_b = _run(b, fb_after, range(F0 + F1), pipeline, hooks={F0 - 1: imp})
    want_b = _run(r, fb, range(F0 + F1), pipeline)
    info = scene_blob_info(packed["blob"])
    assert info["n"] == 3 and list(info["scenes"]) == src
    if not pipeline:                                                 # mmw_pack_results right after the import
        for s, d in MOVES:
            assert packed["b"][d].tobytes() == packed["a"][s].tobytes(), "records of scene %d in slot %d" % (s, d)
    for s, d in MOVES:
        ctx = "frame %d, scene %d in slot %d" % (F0 - 1, s, d)
        if pipeline:                 # the frame's records were produced before the import; the state is the source's
            _same_scene(got_b[F0 - 1][d], got_a[F0 - 1][s], ctx, ("tracks", "summary", "ring", "status"))
            _same_scene(got_b[F0 - 1][d], want_b[F0 - 1][d], ctx, ("results",))
        else:
            _same_scene(got_b[F0 - 1][d], got_a[F0 - 1][s], ctx, STATE_KEYS)
        for f in range(F0, F0 + F1):
            _same_scene(got_b[f][d], got_a[f][s], "frame %d, scene %d in slot %d" % (f, s, d))
    for f in range(F0 + F1):
        for k in range(S1):
            if k not in dst or f < F0 - 1:
                _same_scene(got_b[f][k], want_b[f][k], "frame %d, slot %d" % (f, k))
    assert max(got_a[F0 - 1][s]["summary"][1] for s in src) > 0     # the ids continue from a non-zero next_id
    assert sum(got_a[-1][s]["summary"][0] for s in src) > 0
    return got_a


def test_move_mid_sequence_serial():
    _move_mid_sequence(False)


def test_move_mid_sequence_throughput_mode():
    """The export is queued right after a pipelined step, before that frame's records are read: they are unchanged,
    and the whole run equals the serial one."""
    piped = _move_mid_sequence(True)
    W = _weights()
    serial = _run(_tracker(S1, W), _synth_feeds(0, S1, F0 + F1), range(F0 + F1))
    for f in range(F0 + F1):
        for s in range(S1):
            _same_scene(piped[f][s], serial[f][s], "frame %d scene %d" % (f, s), STATE_KEYS + ("assoc",))


def test_move_to_second_gpu():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _move_mid_sequence(False, device_b=1)


# ---- 3: heterogeneous sensors -----------------------------------------------------------------------------------
S3, F3 = 16, 40
HET_MOVES = ((1, 2), (6, 4), (14, 12))                              # entries differ at each pair
PK_PROFILES = [(16, 0.125, 8), (32, 0.0626, 9), (64, 0.0391, 10)]   # numDopplerBins, dopplerResolutionMps, xyzQFormat


def _packet_feeds(seed, S, F, shift=0):
    """Packets of synthetic scene seed + s, sent by a radar with profile PK_PROFILES[(s + shift) % 3]."""
    out = []
    for s in range(S):
        bins, res, q = PK_PROFILES[(s + shift) % 3]
        sc = synth.gen_scene(seed + s, F, synth.SceneSpec(doppler_res=res))
        out.append([(tlv.encode_packet(f + 1, sc.frames[f], q, res), float(sc.dts()[f])) for f in range(F)])
    return out


@pytest.mark.parametrize("kind", ["fp32", "int16", "packets"])
def test_move_between_heterogeneous_tables(kind):
    W = _weights()
    if kind == "packets":
        fa, fb = _packet_feeds(400, S3, F3), _packet_feeds(450, S3, F3, shift=1)
        ta, tb = ({k: [PK_PROFILES[(s + sh) % 3][i] for s in range(S3)] for i, k in ((0, "num_doppler_bins"),
                                                                                      (1, "doppler_res"))}
                  for sh in (0, 1))
    else:
        pa = [_params(s) for s in range(S3)]
        pb = [_params(s + 5) for s in range(S3)]
        fa = _feeds_from_frames(_frames(range(600, 600 + S3), pa, F3, kind == "int16"))
        fb = _feeds_from_frames(_frames(range(650, 650 + S3), pb, F3, kind == "int16"))
        keys = ("s_height", "s_tilt_deg", "z_max", "doppler_res", "xyz_q_format")
        ta = {k: [p[k] for p in pa] for k in keys}
        tb = {k: [p[k] for p in pb] for k in keys}
    packets = kind == "packets"
    a, b = _tracker(S3, W), _tracker(S3, W)
    a.set_scene_sensors(**{k: np.array(v) for k, v in ta.items()})
    b.set_scene_sensors(**{k: np.array(v) for k, v in tb.items()})
    src = [s for s, _ in HET_MOVES]
    dst = [d for _, d in HET_MOVES]
    assert all(a.scene_sensors()[s].tobytes() != b.scene_sensors()[d].tobytes() for s, d in HET_MOVES)
    blob = {}                        # A runs to the end first: its state at frame F0 - 1 is exported at that frame
    got_a = _run(a, fa, range(F3), hooks={F0 - 1: lambda: blob.update(b=a.export_scenes(src))}, packets=packets)
    got_b = _run(b, _after(fb, F0, [(s, d, fa) for s, d in HET_MOVES]), range(F3),
                 hooks={F0 - 1: lambda: b.import_scenes(blob["b"], dst)}, packets=packets)
    ta_now, tb_now = a.scene_sensors(), b.scene_sensors()
    for s, d in HET_MOVES:
        assert tb_now[d].tobytes() == ta_now[s].tobytes(), "table entry of slot %d" % d
        for f in range(F0, F3):
            _same_scene(got_b[f][d], got_a[f][s], "%s frame %d, scene %d in slot %d" % (kind, f, s, d))
    assert sum(got_a[-1][s]["summary"][0] for s in src) > 0


# ---- 4: round trip ----------------------------------------------------------------------------------------------
def test_round_trip_reproduces_state_dump_and_permutation_continues():
    S, F = 16, 40
    W = _weights()
    feeds = _synth_feeds(800, S, F)
    a, ref = _tracker(S, W), _tracker(S, W)
    _run(a, feeds, range(F0), views=False)
    _run(ref, feeds, range(F0), views=False)
    blob = a.export_scenes(None)
    fresh = _tracker(S, W)
    fresh.import_scenes(blob)
    assert fresh.state_dump().tobytes() == a.state_dump().tobytes()
    perm = np.random.default_rng(5).permutation(S).astype(np.int32)  # scene i -> slot perm[i]
    a.import_scenes(blob, perm)
    moved = [None] * S
    for i in range(S):
        moved[perm[i]] = feeds[i]
    got = _run(a, moved, range(F0, F))
    want = _run(ref, feeds, range(F0, F))
    for k in range(F - F0):
        for i in range(S):
            _same_scene(got[k][perm[i]], want[k][i], "frame %d, scene %d in slot %d" % (F0 + k, i, perm[i]))


# ---- 5: swap ----------------------------------------------------------------------------------------------------
def test_swap_between_contexts():
    S, F = 8, 40
    W = _weights()
    fa, fb = _synth_feeds(900, S, F), _synth_feeds(950, S, F)
    a, b, ra, rb = (_tracker(S, W) for _ in range(4))
    for bt, fd in ((a, fa), (b, fb), (ra, fa), (rb, fb)):
        _run(bt, fd, range(F0), views=False)
    blob_a, blob_b = a.export_scenes([2]), b.export_scenes([5])
    b.import_scenes(blob_a, [5])
    a.import_scenes(blob_b, [2])
    got_a = _run(a, _after(fa, 0, [(5, 2, fb)]), range(F0, F))
    got_b = _run(b, _after(fb, 0, [(2, 5, fa)]), range(F0, F))
    want_a, want_b = _run(ra, fa, range(F0, F)), _run(rb, fb, range(F0, F))
    for k in range(F - F0):
        for s in range(S):
            _same_scene(got_a[k][s], want_b[k][5] if s == 2 else want_a[k][s], "A frame %d slot %d" % (k, s))
            _same_scene(got_b[k][s], want_a[k][2] if s == 5 else want_b[k][s], "B frame %d slot %d" % (k, s))


# ---- 6: full size -----------------------------------------------------------------------------------------------
def test_half_of_a_full_size_context_moves():
    S, F, n = 1024, 30, 512
    W = _weights()
    feeds = _synth_feeds(2000, S, F)
    a, b = _tracker(S, W), _tracker(S, W)
    src = np.arange(1, S, 2, dtype=np.int32)                        # odd scenes -> slots 0 .. 511 of the second context
    dst = np.arange(n, dtype=np.int32)
    _run(a, feeds, range(F0), views=False)
    blob = move_scenes(a, src, b, dst, reset_source=False)
    assert blob.size == b.scene_state_size(n) and scene_blob_info(blob)["n"] == n
    empty = (np.zeros((0, 5), np.float32), 0.083)
    fb = [[empty] * F for _ in range(S)]
    for i in range(n):
        fb[dst[i]] = feeds[src[i]]
    got_a = _run(a, feeds, range(F0, F))
    got_b = _run(b, fb, range(F0, F))
    tracked = 0
    for k in range(F - F0):
        for i in range(n):
            _same_scene(got_b[k][dst[i]], got_a[k][src[i]], "frame %d, scene %d in slot %d" % (F0 + k, src[i], dst[i]))
            tracked += got_a[k][src[i]]["summary"][0]
    assert tracked > 0


# ---- 8: refusals ------------------------------------------------------------------------------------------------
SCENE_OFF = 48                     # record: sensor entry (40 bytes, padded to 48), then the SceneRec


def _layout(ncap, tcap):
    """Offsets of the parts of a scene record, in the library's order (mmw_api.cu, kPart*)."""
    sizes = [64, 1264 * tcap, 3840 * tcap, 60 * ncap, 816, 228 * tcap, 4]
    off, o = [], SCENE_OFF
    for sz in sizes:
        off.append(o)
        o += (sz + 15) // 16 * 16
    return off, o


def _put(blob, at, dtype, value):
    b = blob.copy()
    b[at:at + np.dtype(dtype).itemsize] = np.array([value], dtype).view(np.uint8)
    return b


def test_refusals_change_nothing():
    S, ncap, tcap = 8, 256, 8
    W = _weights()
    feeds = _synth_feeds(1200, S, 20)
    a, b, ref = (_tracker(S, W) for _ in range(3))
    for bt in (a, b, ref):
        bt.set_scene_sensors(doppler_res=[0.0626, 0.125] * 4, num_doppler_bins=[16] * 8)
    a.set_scene_sensors(s_height=[1.2, 1.5, 1.8, 2.1, 2.4, 2.7, 3.0, 3.3])
    _run(a, feeds, range(15), views=False)
    for bt in (b, ref):
        _run(bt, feeds, range(10), views=False)
    lib = a.lib
    n_all = a.summary()[0]
    k2 = int(np.argmax(n_all))                                       # a scene with at least two tracks
    assert n_all[k2] >= 2
    src = np.array([k2, (k2 + 3) % S], np.int32)
    blob = a.export_scenes(src)
    dst = np.array([1, 6], np.int32)
    hs = 64 + 16
    off, rec = _layout(ncap, tcap)
    assert scene_blob_info(blob)["record_bytes"] == rec and blob.size == hs + 2 * rec
    scene0 = hs + off[0]
    track0, track1 = hs + off[1], hs + off[1] + 1264
    sc = np.frombuffer(blob[scene0:scene0 + 64].tobytes(), np.int32)
    n_tracks, slot_mask = int(sc[0]), int(sc[7])
    t0_slot = int(np.frombuffer(blob[track0 + 1228:track0 + 1232].tobytes(), np.int32)[0])
    free_bit = next(k for k in range(tcap) if not slot_mask >> k & 1)
    table = b.scene_sensors().tobytes()
    state = b.state_dump().tobytes()

    def refused(blob_, scenes=dst, n=None, nbytes=None, code=-1):
        scenes = None if scenes is None else np.ascontiguousarray(scenes, np.int32)
        n = len(scenes) if n is None and scenes is not None else n
        rc = lib.mmw_import_scenes(b._h, _lib.ptr(scenes), n, _lib.ptr(blob_), blob_.size if nbytes is None else nbytes)
        assert rc == code, (rc, lib.mmw_last_error())

    bad = {
        "magic": _put(blob, 0, "<u4", 0x4D4D5753), "abi": _put(blob, 4, "<u4", 6),
        "ncap": _put(blob, 12, "<i4", 128), "tcap": _put(blob, 16, "<i4", 16), "frames_batch": _put(blob, 20, "<i4", 0),
        "header n": _put(blob, 8, "<i4", 1), "record_bytes": _put(blob, 24, "<u8", rec + 16),
        "total_bytes": _put(blob, 32, "<u8", blob.size + 16),
        "n_tracks > tcap": _put(blob, scene0, "<i4", tcap + 1), "n_tracks < 0": _put(blob, scene0, "<i4", -1),
        "ring_n": _put(blob, scene0 + 8, "<i4", 4), "ring_n < 0": _put(blob, scene0 + 8, "<i4", -1),
        "ring_head": _put(blob, scene0 + 12, "<i4", 3), "ring_head < 0": _put(blob, scene0 + 12, "<i4", -1),
        "ring_cnt": _put(blob, scene0 + 16, "<i4", ncap + 1), "ring_cnt < 0": _put(blob, scene0 + 24, "<i4", -1),
        "slot_mask spare bit": _put(blob, scene0 + 28, "<u4", slot_mask | 1 << free_bit),
        "slot_mask above tcap": _put(blob, scene0 + 28, "<u4", slot_mask | 1 << tcap),
        "slot_mask missing bit": _put(blob, scene0 + 28, "<u4", slot_mask & ~(1 << t0_slot)),
        "track slot >= tcap": _put(blob, track0 + 1228, "<i4", tcap),
        "track slot < 0": _put(blob, track0 + 1228, "<i4", -1),
        "track slots alike": _put(blob, track1 + 1228, "<i4", t0_slot),
        "track slot outside mask": _put(blob, track0 + 1228, "<i4", free_bit),
        "track ring_n": _put(blob, track1 + 1232, "<i4", 4), "track ring_head": _put(blob, track1 + 1236, "<i4", 3),
        "track ring_cnt": _put(blob, track1 + 1240, "<i4", 65), "track ring_cnt < 0": _put(blob, track0 + 1248, "<i4", -1),
        "pose_cnt": _put(blob, hs + off[6], "<i4", tcap + 1), "pose_cnt < 0": _put(blob, hs + off[6], "<i4", -1),
        "doppler_res 0": _put(blob, hs + 24, "<f8", 0.0), "q format": _put(blob, hs + 32, "<i4", 16),
        "height nan": _put(blob, hs, "<f8", np.nan), "num_doppler_bins": _put(blob, hs + 36, "<i4", -1),
        "second record": _put(blob, hs + rec + off[0], "<i4", tcap + 1),
    }
    assert n_tracks >= 2
    for name, bb in bad.items():
        assert bb.tobytes() != blob.tobytes(), name
        refused(bb)
    refused(blob, nbytes=blob.size - 1)                             # truncated
    refused(blob, nbytes=10)
    refused(blob, scenes=dst[:1])                                    # n differs from the blob's
    refused(blob, scenes=[1, 1])
    refused(blob, scenes=[1, 8])
    refused(blob, scenes=[-1, 2])
    refused(blob, scenes=None, n=2)
    refused(blob, n=-1)
    assert lib.mmw_import_scenes(b._h, _lib.ptr(dst), 2, None, blob.size) == -1
    # export: bad lists, NULL pointers, a buffer too small
    out = np.zeros(blob.size, np.uint8)
    for idx in ([0, 0], [8], [-1]):
        i = np.array(idx, np.int32)
        assert lib.mmw_export_scenes(b._h, _lib.ptr(i), i.size, _lib.ptr(out), out.size) == -1, idx
    assert lib.mmw_export_scenes(b._h, None, 2, _lib.ptr(out), out.size) == -1
    assert lib.mmw_export_scenes(b._h, _lib.ptr(dst), 2, None, out.size) == -1
    assert lib.mmw_export_scenes(b._h, _lib.ptr(dst), -1, _lib.ptr(out), out.size) == -1
    assert lib.mmw_export_scenes(b._h, _lib.ptr(dst), 2, _lib.ptr(out), out.size - 1) == -3
    # n = 0: a header-only blob, a no-op import
    empty = b.export_scenes([])
    assert empty.size == 64 and scene_blob_info(empty)["n"] == 0
    b.import_scenes(empty, [])
    assert b.scene_sensors().tobytes() == table
    assert b.state_dump().tobytes() == state
    got = _run(b, feeds, range(10, 15))
    want = _run(ref, feeds, range(10, 15))
    assert got == want
    # the unmodified blob is accepted
    b.import_scenes(blob, dst)
    assert b.scene_sensors()[dst].tobytes() == a.scene_sensors()[src].tobytes()
