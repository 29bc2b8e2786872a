"""Batched host API: S independent scenes on one GPU, stepped one radar frame at a time.

This is the call a user of the batched path makes; it is a thin layer over the C ABI
(include/mmw.h) and does no arithmetic of its own.  The single-scene drop-in façade that mirrors
the reference's ``Tracking.TrackBuffer`` / ``Utils.normalize_data`` names sits on top of it in
``mmwave_msc_b200/Tracking.py`` and ``Utils.py``.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from . import pose_weights as pw


def default_config(**overrides) -> _lib.Config:
    """mmw_config filled with the reference's constants.py defaults; keyword overrides by field name
    (e.g. ``tr_max_tracks=10``, ``frames_batch=0``)."""
    cfg = _lib.Config()
    _lib.check(_lib.load().mmw_default_config(C.byref(cfg)))
    for k, v in overrides.items():
        if k == "kf_spread_lim":
            for i, x in enumerate(v):
                cfg.kf_spread_lim[i] = float(x)
        elif k == "default_posture":
            for i, x in enumerate(v):
                cfg.default_posture[i] = float(x)
        else:
            if not hasattr(cfg, k):
                raise AttributeError("mmw_config has no field %r" % k)
            setattr(cfg, k, v)
    return cfg


def config_from_constants(const) -> _lib.Config:
    """Builds mmw_config from a module shaped like the reference's ``constants`` (constants.py)."""
    if getattr(const, "MOTION_MODEL", None) is not None and getattr(const.MOTION_MODEL, "KF_DIM", [9, 6])[0] != 9:
        raise NotImplementedError("only MOTION_MODEL = CONST_ACC_MODEL (constants.py:246) is implemented")
    return default_config(
        s_height=float(const.S_HEIGHT), s_tilt_deg=float(const.S_TILT), frames_batch=int(const.FB_FRAMES_BATCH),
        db_min_samples=int(const.DB_MIN_SAMPLES_MIN), db_z_weight=float(const.DB_Z_WEIGHT),
        db_range_weight=float(const.DB_RANGE_WEIGHT), db_eps=float(const.DB_EPS),
        tr_max_tracks=int(const.TR_MAX_TRACKS), kf_enable_est=int(bool(const.KF_ENABLE_EST)),
        tr_lifetime_dynamic=float(const.TR_LIFETIME_DYNAMIC), tr_lifetime_static=float(const.TR_LIFETIME_STATIC),
        tr_vel_thres=float(const.TR_VEL_THRES), tr_gate=float(const.TR_GATE), kf_q_var=float(const.KF_Q_STD),
        kf_p_init=float(const.KF_P_INIT), kf_group_disp_init=float(const.KF_GROUP_DISP_EST_INIT),
        kf_a_n=float(const.KF_A_N), kf_a_spr=float(const.KF_A_SPR), kf_spread_lim=list(const.KF_SPREAD_LIM),
        kf_est_pointnum=int(const.KF_EST_POINTNUM), intensity_mu=float(const.INTENSITY_MU),
        intensity_std=float(const.INTENSITY_STD), default_posture=list(np.asarray(const.MODEL_DEFAULT_POSTURE)),
        m_x=float(getattr(const, "M_X", 0.32)), m_y=float(getattr(const, "M_Y", -0.6)),
        m_z=float(getattr(const, "M_Z", 1.3)), fade_size_max=float(getattr(const, "V_SCREEN_FADE_SIZE_MAX", 0.3)),
        fade_size_min=float(getattr(const, "V_SCREEN_FADE_SIZE_MIN", 0.2)),
        fade_weight=float(getattr(const, "V_SCREEN_FADE_WEIGHT", 0.08)),
        doppler_res=float(getattr(const, "DOPPLER_RESOLUTION", None) or 1.0))


def concat_packets(packets: Sequence[Optional[bytes]]) -> Tuple[np.ndarray, np.ndarray]:
    """One framed UART packet (bytes) or None per scene -> (blob (bytes,) uint8, offsets (S+1,) int64), the layout
    ``BatchedTracker.step_packets`` takes: scene s's packet is blob[offsets[s]:offsets[s+1]], empty for None."""
    parts = [b"" if p is None else bytes(p) for p in packets]
    offsets = np.zeros(len(parts) + 1, np.int64)
    offsets[1:] = np.cumsum([len(p) for p in parts])
    return np.frombuffer(b"".join(parts), dtype=np.uint8).copy(), offsets


def scene_blob_info(blob) -> dict:
    """Header and source scene indices of a scene blob (``BatchedTracker.export_scenes``), read on the host: n,
    abi_version, max_points_per_frame, max_tracks, frames_batch, record_bytes, total_bytes and scenes ((n,) int32).
    ValueError for a blob that is not a scene blob or is shorter than its header says."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8).reshape(-1)
    hs = C.sizeof(_lib.SceneBlobHeader)
    if blob.size < hs:
        raise ValueError("scene blob is truncated: %d bytes, the header alone has %d" % (blob.size, hs))
    h = _lib.SceneBlobHeader.from_buffer_copy(blob[:hs].tobytes())
    if h.magic != _lib.SCENE_BLOB_MAGIC:
        raise ValueError("not a scene blob (magic 0x%08x)" % h.magic)
    if h.n < 0 or blob.size < h.total_bytes or h.total_bytes < hs + (4 * h.n + 15) // 16 * 16 + h.n * h.record_bytes:
        raise ValueError("scene blob is truncated or its sizes are inconsistent")
    info = {k: int(getattr(h, k)) for k in ("n", "abi_version", "max_points_per_frame", "max_tracks", "frames_batch",
                                            "record_bytes", "total_bytes")}
    info["scenes"] = blob[hs:hs + 4 * h.n].view(np.int32).copy()
    return info


class BatchedTracker:
    """S scenes resident on one GPU.  ``step`` = the loop body of the reference's offline_main.py:45-60
    for every scene at once."""

    def __init__(self, n_scenes: int, max_points: int = 256, max_tracks: int = 8, device: int = 0,
                 config: Optional[_lib.Config] = None):
        self.lib = _lib.load()
        self.cfg = config if config is not None else default_config()
        self.S, self.ncap, self.tcap, self.device = int(n_scenes), int(max_points), int(max_tracks), int(device)
        h = C.c_void_p()
        _lib.check(self.lib.mmw_create(C.byref(self.cfg), self.device, self.S, self.ncap, self.tcap, C.byref(h)))
        self._h = h
        self._n_last = 0
        self.pose_variant: Optional[int] = None

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.mmw_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        _lib.check(self.lib.mmw_reset(self._h))

    def set_doppler_resolution(self, doppler_res: float):
        """Unit of the Doppler column of the point rows: doppler [m/s] = row[3] * doppler_res in float64 on the device
        (mmw_config::doppler_res).  With the sensor's dopplerResolutionMps the rows carry dopplerIdx.  Sets the unit of
        every scene."""
        _lib.check(self.lib.mmw_set_doppler_resolution(self._h, float(doppler_res)))
        self.cfg.doppler_res = float(doppler_res)

    # -- per-scene sensors --------------------------------------------------------------------------
    def _scene_index(self, scenes) -> np.ndarray:
        if scenes is None or isinstance(scenes, slice):
            return np.arange(self.S, dtype=np.int32)[scenes if scenes is not None else slice(None)]
        return np.ascontiguousarray(np.atleast_1d(scenes), dtype=np.int32).reshape(-1)

    def scene_sensors(self) -> np.ndarray:
        """Every scene's sensor mounting and radar profile (mmw_scene_sensor): a (S,) structured array
        (``_lib.SCENE_SENSOR_DTYPE``) with s_height, s_tilt_deg, z_max, doppler_res, xyz_q_format, num_doppler_bins."""
        out = np.zeros(self.S, _lib.SCENE_SENSOR_DTYPE)
        _lib.check(self.lib.mmw_get_scene_sensors(self._h, 0, self.S, _lib.ptr(out)))
        return out

    def set_scene_sensors(self, s_height=None, s_tilt_deg=None, z_max=None, doppler_res=None, xyz_q_format=None,
                          scenes=None, num_doppler_bins=None):
        """Sets the mounting and radar profile of the selected scenes (``scenes``: a slice or index array, default all).
        Each value is a scalar or an array with one entry per selected scene; None keeps the current value.  Takes
        effect with the next step.  Rows already in a scene's rings are re-read under the new values: change a scene
        before its first frame, or together with ``reset_scenes``.  All or nothing: invalid values change no scene.
        ``num_doppler_bins`` is the radar profile's numDopplerBins, which ``step_packets`` needs (with ``doppler_res`` =
        the profile's dopplerResolutionMps)."""
        idx = self._scene_index(scenes)
        table = self.scene_sensors()
        for name, v in (("s_height", s_height), ("s_tilt_deg", s_tilt_deg), ("z_max", z_max),
                        ("doppler_res", doppler_res), ("xyz_q_format", xyz_q_format),
                        ("num_doppler_bins", num_doppler_bins)):
            if v is None:
                continue
            v = np.asarray(v)
            if v.ndim and v.shape != idx.shape:
                raise ValueError("%s: give a scalar or one value per selected scene" % name)
            if name in ("xyz_q_format", "num_doppler_bins") and not np.array_equal(v, np.round(v)):
                raise ValueError("%s must be an integer" % name)
            table[name][idx] = v
        _lib.check(self.lib.mmw_set_scene_sensors(self._h, 0, self.S, _lib.ptr(table)))

    def reset_scenes(self, scenes):
        """``reset`` restricted to the selected scenes (a slice or index array): their tracks, rings and id counters
        start afresh; other scenes and the sensor table are left alone."""
        idx = self._scene_index(scenes)
        _lib.check(self.lib.mmw_reset_scenes(self._h, _lib.ptr(idx), idx.size))

    @property
    def stream(self) -> int:
        """cudaStream_t of the context as an integer (e.g. for torch.cuda.ExternalStream)."""
        return int(self.lib.mmw_stream(self._h) or 0)

    # -- pose weights -----------------------------------------------------------------------------
    def load_pose_weights(self, weights: Sequence[np.ndarray], variant: Optional[int] = None):
        if variant is None:
            variant = pw.VARIANT_3D if self.cfg.frames_batch == 2 else pw.VARIANT_2D
        blob = pw.pack_blob(list(weights))
        _lib.check(self.lib.mmw_load_pose_weights(self._h, int(variant), _lib.ptr(blob), blob.size))
        self.pose_variant = int(variant)

    def set_dense_path(self, tensor_cores: bool):
        _lib.check(self.lib.mmw_set_dense_path(self._h, 1 if tensor_cores else 0))

    def pose_intermediate(self, layer: int, tensor_cores: bool = True):
        """Test hook: layer 0..3 of the last serial pose-network run (include/mmw.h, mmw_pose_intermediate), one row per
        pose row, values in Keras order.  Tensor-core path: (hi, lo) uint16 arrays of the raw bf16 bits; CUDA-core path
        (``tensor_cores=False``, layers 2 and 3): float32."""
        n = C.c_int(0)
        _lib.check(self.lib.mmw_pose_intermediate(self._h, int(layer), C.byref(n), None, 0))
        D = self.cfg.frames_batch + 1
        per = [D * 64 * 5, D * 64 * 16, D * 64 * 32, D * 512][layer]
        out = np.zeros((2, n.value, per) if tensor_cores else (n.value, per), np.uint16 if tensor_cores else np.float32)
        _lib.check(self.lib.mmw_pose_intermediate(self._h, int(layer), C.byref(n), _lib.ptr(out), out.nbytes))
        return (out[0], out[1]) if tensor_cores else out

    # -- the hot path -----------------------------------------------------------------------------
    def step(self, points: np.ndarray, offsets: np.ndarray, dt: np.ndarray, pose: bool = True,
             record_labels: bool = False, pipeline: bool = False):
        """Host inputs: points (sum N, 5) float32, offsets (S+1,) int32, dt (S,) float64.
        ``pipeline`` (throughput mode, MMW_STEP_PIPELINE): this frame's pose network overlaps the next frame's tracker;
        fetch the frame's results with read_results_async() right after the call."""
        i16 = getattr(points, "dtype", None) == np.int16         # the sensor's lattice: x, y, z, dopplerIdx, peakVal
        points = np.ascontiguousarray(points, dtype=np.int16 if i16 else np.float32).reshape(-1, 5)
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        if offsets.shape != (self.S + 1,) or dt.shape != (self.S,):
            raise ValueError("offsets must have S+1 entries and dt S entries")
        if int(offsets[-1]) != points.shape[0]:
            raise ValueError("offsets[-1] must equal the number of point rows")
        flags = ((_lib.STEP_POSE if pose else 0) | (_lib.STEP_RECORD_LABELS if record_labels else 0) |
                 (_lib.STEP_PIPELINE if pipeline else 0) | (_lib.STEP_INPUT_I16 if i16 else 0))
        self._n_last = points.shape[0]
        _lib.check(self.lib.mmw_step(self._h, _lib.ptr(points), _lib.ptr(offsets), _lib.ptr(dt), flags))

    def step_packets(self, blob: np.ndarray, offsets: np.ndarray, dt: np.ndarray, pose: bool = True,
                     record_labels: bool = False, pipeline: bool = False) -> Tuple[np.ndarray, np.ndarray]:
        """One frame for every scene from its sensor's UART packet (mmw_step_packets): ReadIWR14xx.read() on the
        device, with each scene's own num_doppler_bins (``set_scene_sensors``), then ``step``.  blob (bytes,) uint8 and
        offsets (S+1,) int64 as ``concat_packets`` builds them, dt (S,) float64.  Returns (frame_numbers (S,) int32,
        data_ok (S,) bool); a scene without a packet or with dataOK = 0 is skipped this frame.  Asynchronous when blob
        is pinned memory; keep it unchanged until the next-but-one step."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8).reshape(-1)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        dt = np.ascontiguousarray(dt, dtype=np.float64)
        if offsets.shape != (self.S + 1,) or dt.shape != (self.S,):
            raise ValueError("offsets must have S+1 entries and dt S entries")
        if int(offsets[0]) != 0 or int(offsets[-1]) > blob.size:
            raise ValueError("offsets must start at 0 and end within the blob")
        flags = ((_lib.STEP_POSE if pose else 0) | (_lib.STEP_RECORD_LABELS if record_labels else 0) |
                 (_lib.STEP_PIPELINE if pipeline else 0))
        frames = np.zeros(self.S, np.int32)
        ok = np.zeros(self.S, np.int32)
        _lib.check(self.lib.mmw_step_packets(self._h, _lib.ptr(blob), _lib.ptr(offsets), _lib.ptr(dt), flags,
                                             _lib.ptr(frames), _lib.ptr(ok)))
        # rows of the step (for point_assoc): numObj (u16 at byte 44) of every packet that yielded objects
        at = offsets[:-1][ok != 0] + 44
        self._n_last = int((blob[at].astype(np.int64) | (blob[at + 1].astype(np.int64) << 8)).sum())
        return frames, ok.astype(bool)

    def step_device(self, points_ptr: int, offsets_ptr: int, dt_ptr: int, n_points: int, pose: bool = True,
                    pipeline: bool = False):
        """Inputs already resident in HBM (device pointers, same layouts as ``step``)."""
        flags = _lib.STEP_DEVICE_INPUT | (_lib.STEP_POSE if pose else 0) | (_lib.STEP_PIPELINE if pipeline else 0)
        self._n_last = int(n_points)
        _lib.check(self.lib.mmw_step(self._h, C.c_void_p(points_ptr), C.c_void_p(offsets_ptr), C.c_void_p(dt_ptr),
                                     flags))

    def run_frames(self, points: np.ndarray, frame_row_offsets: np.ndarray, offsets: np.ndarray, dt: np.ndarray,
                   results: np.ndarray, pose: bool = True, pipeline: bool = True, n_records: Optional[np.ndarray] = None):
        """F frames back to back from host buffers, the loop in C (mmw_run_frames): points (rows, 5) float32 or int16,
        frame_row_offsets (F+1,) int64, offsets (F, S+1) int32 (each frame's own, starting at 0), dt (F, S) float64,
        results (F, S * max_tracks * 72) float32 filled with every frame's packed records.  Blocking.
        With ``n_records`` ((F,) int32; it and ``results`` in pinned memory) only the live tracks' records come back
        (mmw_run_frames_compact): frame f's first n_records[f] records, field 71 = scene index; see
        ``expand_compact_results``."""
        i16 = points.dtype == np.int16
        F = len(frame_row_offsets) - 1
        for a, dt_, shp in ((points, np.int16 if i16 else np.float32, None), (frame_row_offsets, np.int64, (F + 1,)),
                            (offsets, np.int32, (F, self.S + 1)), (dt, np.float64, (F, self.S)),
                            (results, np.float32, (F, self.S * self.tcap * _lib.RESULT_FLOATS))):
            if a.dtype != dt_ or not a.flags["C_CONTIGUOUS"] or (shp is not None and a.shape != shp):
                raise ValueError("run_frames: wrong dtype / shape / layout of an argument")
        flags = ((_lib.STEP_POSE if pose else 0) | (_lib.STEP_PIPELINE if pipeline else 0) |
                 (_lib.STEP_INPUT_I16 if i16 else 0))
        if n_records is not None:
            if n_records.dtype != np.int32 or n_records.shape != (F,) or not n_records.flags["C_CONTIGUOUS"]:
                raise ValueError("run_frames: n_records must be a contiguous int32 array with one entry per frame")
            _lib.check(self.lib.mmw_run_frames_compact(self._h, F, _lib.ptr(points), _lib.ptr(frame_row_offsets),
                                                       _lib.ptr(offsets), _lib.ptr(dt), _lib.ptr(results),
                                                       _lib.ptr(n_records), flags))
        else:
            _lib.check(self.lib.mmw_run_frames(self._h, F, _lib.ptr(points), _lib.ptr(frame_row_offsets),
                                               _lib.ptr(offsets), _lib.ptr(dt), _lib.ptr(results), flags))
        self._n_last = int(frame_row_offsets[-1] - frame_row_offsets[-2]) if F else 0

    def expand_compact_results(self, frame_block: np.ndarray, n: int) -> np.ndarray:
        """The full (S, max_tracks, 72) record array of a frame from its compact block (run_frames with n_records):
        empty slots get id -1 and the scene's track count, like mmw_pack_results writes them."""
        R = _lib.RESULT_FLOATS
        rec = np.asarray(frame_block[:n * R], np.float32).reshape(n, R)
        out = np.zeros((self.S, self.tcap, R), np.float32)
        out[:, :, 0] = -1.0
        if n:
            scene = rec[:, R - 1].astype(np.int64)
            first = np.r_[True, scene[1:] != scene[:-1]]
            start = np.maximum.accumulate(np.where(first, np.arange(n), 0))
            k = np.arange(n) - start
            out[scene, k] = rec
            out[scene, k, R - 1] = 0.0
            out[scene, :, 1] = rec[:, 1][:, None]
        return out

    def estimate_posture(self):
        """TrackBuffer.estimate_posture alone (needs load_pose_weights first)."""
        _lib.check(self.lib.mmw_estimate_posture(self._h))

    def pose_features_only(self):
        _lib.check(self.lib.mmw_pose_features_only(self._h))

    def set_keypoints(self, scene: int, track_index: int, kp: np.ndarray):
        kp = np.ascontiguousarray(kp, dtype=np.float32).reshape(57)
        _lib.check(self.lib.mmw_set_keypoints(self._h, int(scene), int(track_index), _lib.ptr(kp)))

    def read_results_async(self, host_out: np.ndarray) -> int:
        """Queues pack + download of the current results into ``host_out`` (float32, S*max_tracks*68, ideally
        pinned) without blocking; returns the slot to hand to ``wait_results``."""
        if host_out.dtype != np.float32 or host_out.size != self.S * self.tcap * _lib.RESULT_FLOATS:
            raise ValueError("host_out must be float32 with S*max_tracks*%d elements" % _lib.RESULT_FLOATS)
        slot = C.c_int(0)
        _lib.check(self.lib.mmw_read_results_async(self._h, _lib.ptr(host_out), C.byref(slot)))
        return slot.value

    def wait_results(self, slot: int):
        _lib.check(self.lib.mmw_wait_results(self._h, int(slot)))

    def sync(self):
        _lib.check(self.lib.mmw_sync(self._h))

    # -- readback ---------------------------------------------------------------------------------
    def tracks(self) -> Tuple[np.ndarray, np.ndarray]:
        """(records, n_tracks): records is a (S, max_tracks) structured array (``_lib.TRACK_DTYPE``) in
        effective_tracks list order; entries >= n_tracks[s] have id == -1."""
        rec = np.zeros((self.S, self.tcap), dtype=_lib.TRACK_DTYPE)
        n = np.zeros(self.S, dtype=np.int32)
        _lib.check(self.lib.mmw_get_tracks(self._h, _lib.ptr(rec), _lib.ptr(n)))
        return rec, n

    def summary(self):
        n = np.zeros(self.S, np.int32); nid = np.zeros(self.S, np.int32); m = np.zeros(self.S, np.int32)
        _lib.check(self.lib.mmw_get_scene_summary(self._h, _lib.ptr(n), _lib.ptr(nid), _lib.ptr(m)))
        return n, nid, m

    def point_assoc(self) -> np.ndarray:
        a = np.zeros(self._n_last, dtype=np.int32)
        if self._n_last:
            _lib.check(self.lib.mmw_get_point_assoc(self._h, _lib.ptr(a), a.size))
        return a

    def labels(self) -> Tuple[np.ndarray, np.ndarray]:
        lab = np.zeros((self.S, 3 * self.ncap), dtype=np.int32)
        n = np.zeros(self.S, dtype=np.int32)
        _lib.check(self.lib.mmw_get_labels(self._h, _lib.ptr(lab), _lib.ptr(n)))
        return lab, n

    def status(self) -> np.ndarray:
        f = np.zeros(self.S, dtype=np.uint32)
        _lib.check(self.lib.mmw_get_status(self._h, _lib.ptr(f)))
        return f

    def ring_counts(self) -> np.ndarray:
        c = np.zeros((self.S, 3), dtype=np.int32)
        _lib.check(self.lib.mmw_get_ring_counts(self._h, _lib.ptr(c)))
        return c

    def ring_pop(self, scene: int = 0):
        _lib.check(self.lib.mmw_ring_pop(self._h, int(scene)))

    def ring_clear(self, scene: int = 0):
        _lib.check(self.lib.mmw_ring_clear(self._h, int(scene)))

    def pose_rows(self, with_features: bool = True):
        """(scene_idx, track_idx, feats) of the last pose batch; feats (rows, frames, 8, 8, 5) float32."""
        n = C.c_int32(0)
        _lib.check(self.lib.mmw_get_pose_rows(self._h, C.byref(n), None, None, None, 0))
        rows = n.value
        nfr = self.cfg.frames_batch + 1
        si = np.zeros(rows, np.int32); ti = np.zeros(rows, np.int32)
        feats = np.zeros((rows, nfr, 8, 8, 5), np.float32) if with_features else None
        if rows:
            _lib.check(self.lib.mmw_get_pose_rows(self._h, C.byref(n), _lib.ptr(si), _lib.ptr(ti),
                                                  _lib.ptr(feats) if with_features else None,
                                                  feats.size if with_features else 0))
        if feats is not None and nfr == 1:
            feats = feats.reshape(rows, 8, 8, 5)
        return si, ti, feats

    def counters(self, reset: bool = False) -> np.ndarray:
        out = np.zeros(8, dtype=np.uint64)
        _lib.check(self.lib.mmw_get_counters(self._h, _lib.ptr(out), 1 if reset else 0))
        return out

    def profile_kernels(self, step_fn, n_steps: int) -> dict:
        """Average device milliseconds per launch of each kernel class over n_steps calls of step_fn(i)
        (CUDA events on the library's stream around every launch; not a profiler run)."""
        _lib.check(self.lib.mmw_profile(self._h, 1))
        for i in range(n_steps):
            step_fn(i)
        ms = np.zeros(8, np.float64); calls = np.zeros(8, np.uint64)
        _lib.check(self.lib.mmw_get_kernel_ms(self._h, _lib.ptr(ms), _lib.ptr(calls)))
        _lib.check(self.lib.mmw_profile(self._h, 0))
        return {_lib.KERNEL_NAMES[i]: float(ms[i] / calls[i]) for i in range(8) if calls[i] > 0}

    def launch_count(self) -> int:
        return int(self.lib.mmw_launch_count(self._h))

    def decode_tlv(self, packets, num_doppler_bins: float, doppler_res: float):
        """Framed xWR14xx UART packets (list of bytes) -> (points (sum N, 5) float32, offsets (n+1,) int32,
        frame_numbers (n,), data_ok (n,) bool): ReadIWR14xx.read's decode of each packet (ReadDataIWR1443.py:88-201),
        in the ragged layout step() takes."""
        n = len(packets)
        offs = np.zeros(n + 1, np.int64)
        offs[1:] = np.cumsum([len(p) for p in packets])
        blob = np.frombuffer(b"".join(packets), dtype=np.uint8) if offs[-1] else np.zeros(1, np.uint8)
        cap = int(max(0, (int(offs[-1]) - 48 * n) // 12 + n))          # 12 bytes per object after the headers
        points = np.zeros((max(cap, 1), 5), np.float32)
        poff = np.zeros(n + 1, np.int32)
        frames = np.zeros(max(n, 1), np.int32)
        ok = np.zeros(max(n, 1), np.int32)
        _lib.check(self.lib.mmw_decode_tlv(self._h, _lib.ptr(np.ascontiguousarray(blob)), _lib.ptr(offs), n,
                                           float(num_doppler_bins), float(doppler_res), _lib.ptr(points),
                                           points.shape[0], _lib.ptr(poff), _lib.ptr(frames), _lib.ptr(ok)))
        return points[:poff[-1]], poff, frames[:n], ok[:n].astype(bool)

    def state_dump(self) -> np.ndarray:
        """Tracker state of all scenes as one uint8 blob (mmw_state_dump): checkpoint of a replay."""
        blob = np.zeros(int(self.lib.mmw_state_size(self._h)), np.uint8)
        _lib.check(self.lib.mmw_state_dump(self._h, _lib.ptr(blob), blob.size))
        return blob

    def state_restore(self, blob: np.ndarray):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        _lib.check(self.lib.mmw_state_restore(self._h, _lib.ptr(blob), blob.size))

    def scene_state_size(self, n: int) -> int:
        """Bytes of a scene blob of n scenes of this context's shape (mmw_scene_state_size)."""
        return int(self.lib.mmw_scene_state_size(self._h, int(n)))

    def export_scenes(self, scenes, out: Optional[np.ndarray] = None) -> np.ndarray:
        """Tracker state and sensor-table entry of the selected scenes (a slice or index array) as one uint8 scene blob
        (mmw_export_scenes); the scenes are left unchanged.  ``out``: a contiguous uint8 buffer of at least
        ``scene_state_size(n)`` bytes to write into (e.g. pinned memory); the blob is its head."""
        idx = self._scene_index(scenes)
        need = self.scene_state_size(idx.size)
        if out is None:
            out = np.empty(need, np.uint8)
        elif out.dtype != np.uint8 or out.ndim != 1 or not out.flags["C_CONTIGUOUS"]:
            raise ValueError("out must be a contiguous 1-D uint8 array")
        _lib.check(self.lib.mmw_export_scenes(self._h, _lib.ptr(idx), idx.size, _lib.ptr(out), out.size))
        return out[:need]

    def import_scenes(self, blob: np.ndarray, scenes=None):
        """Puts the scenes of a scene blob into the selected slots (a slice or index array, one per scene of the blob;
        default: the blob's own source indices), sensor-table entries included (mmw_import_scenes).  Their tracks
        continue where the exported ones left off.  A malformed blob changes nothing (MmwError)."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8).reshape(-1)
        idx = scene_blob_info(blob)["scenes"] if scenes is None else self._scene_index(scenes)
        _lib.check(self.lib.mmw_import_scenes(self._h, _lib.ptr(idx), idx.size, _lib.ptr(blob), blob.size))

    def export_track0(self):
        """Dataset-builder export (preprocessing.py:185-216): (rows [S,192,5] float64, valid [S] bool,
        centroid [S,2]) of track 0 of every scene after the last step."""
        rows = np.zeros((self.S, 192, 5), np.float64)
        valid = np.zeros(self.S, np.int32)
        cen = np.zeros((self.S, 2), np.float64)
        _lib.check(self.lib.mmw_export_track0(self._h, _lib.ptr(rows), _lib.ptr(valid), _lib.ptr(cen)))
        return rows, valid.astype(bool), cen

    def pack_results(self, device_ptr: int):
        _lib.check(self.lib.mmw_pack_results(self._h, C.c_void_p(device_ptr)))

    # -- stage-level entry points (known-answer tests) ------------------------------------------------
    def preprocess(self, points: np.ndarray):
        points = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 5)
        world = np.zeros((points.shape[0], 8), np.float64)
        keep = np.zeros(points.shape[0], np.uint8)
        _lib.check(self.lib.mmw_preprocess(self._h, _lib.ptr(points), points.shape[0], _lib.ptr(world),
                                           _lib.ptr(keep)))
        return world, keep.astype(bool)

    def dbscan(self, clouds: List[np.ndarray], eps: float = 0.0, min_samples: int = 0) -> List[np.ndarray]:
        counts = [len(c) for c in clouds]
        offsets = np.zeros(len(clouds) + 1, np.int32)
        offsets[1:] = np.cumsum(counts)
        xyz = (np.concatenate([np.asarray(c, np.float64)[:, :3] for c in clouds], axis=0)
               if sum(counts) else np.zeros((0, 3)))
        xyz = np.ascontiguousarray(xyz, dtype=np.float64)
        labels = np.full(int(offsets[-1]), -9, np.int32)
        _lib.check(self.lib.mmw_dbscan(self._h, _lib.ptr(xyz), _lib.ptr(offsets), len(clouds), float(eps),
                                       int(min_samples), _lib.ptr(labels)))
        return [labels[offsets[i]:offsets[i + 1]] for i in range(len(clouds))]

    def kalman_predict(self, x: np.ndarray, P: np.ndarray, dt: np.ndarray):
        x = np.ascontiguousarray(x, np.float64).reshape(-1, 9).copy()
        P = np.ascontiguousarray(P, np.float64).reshape(-1, 81).copy()
        dt = np.ascontiguousarray(dt, np.float64)
        _lib.check(self.lib.mmw_kalman_predict(self._h, _lib.ptr(x), _lib.ptr(P), _lib.ptr(dt), x.shape[0]))
        return x, P.reshape(-1, 9, 9)

    def kalman_update(self, x, P, z, R, lifetime_is_zero):
        x = np.ascontiguousarray(x, np.float64).reshape(-1, 9).copy()
        P = np.ascontiguousarray(P, np.float64).reshape(-1, 81).copy()
        z = np.ascontiguousarray(z, np.float64).reshape(-1, 6)
        R = np.ascontiguousarray(R, np.float64).reshape(-1, 36)
        l0 = np.ascontiguousarray(lifetime_is_zero, np.uint8)
        _lib.check(self.lib.mmw_kalman_update(self._h, _lib.ptr(x), _lib.ptr(P), _lib.ptr(z), _lib.ptr(R),
                                              _lib.ptr(l0), x.shape[0]))
        return x, P.reshape(-1, 9, 9)

    def gate(self, points6: np.ndarray, hx: np.ndarray, Cmat: np.ndarray):
        pts = np.ascontiguousarray(points6, np.float64).reshape(-1, 6)
        hx = np.ascontiguousarray(hx, np.float64).reshape(-1, 6)
        Cm = np.ascontiguousarray(Cmat, np.float64).reshape(-1, 36)
        T = hx.shape[0]
        d2 = np.zeros((pts.shape[0], max(T, 1)), np.float64)
        assoc = np.zeros(pts.shape[0], np.int32)
        _lib.check(self.lib.mmw_gate(self._h, _lib.ptr(pts), pts.shape[0], _lib.ptr(hx), _lib.ptr(Cm), T,
                                     _lib.ptr(d2), _lib.ptr(assoc)))
        return d2[:, :T], assoc

    def pose(self, feats: np.ndarray) -> np.ndarray:
        feats = np.ascontiguousarray(feats, np.float32)
        n = feats.shape[0]
        per = (self.cfg.frames_batch + 1) * 64 * 5
        if feats.size != n * per:
            raise ValueError("feature maps must have %d values per row" % per)
        out = np.zeros((n, 57), np.float32)
        _lib.check(self.lib.mmw_pose(self._h, _lib.ptr(feats), n, _lib.ptr(out)))
        return out


def _phase_clocks(self, enable: bool):
    """Debug: cycles per phase of the fused step kernel accumulated since the last call (16 counters)."""
    out = np.zeros(16, dtype=np.uint64)
    _lib.check(self.lib.mmw_phase_clocks(self._h, 1 if enable else 0, _lib.ptr(out)))
    return out


BatchedTracker.phase_clocks = _phase_clocks
