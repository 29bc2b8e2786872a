/*
 * mmw.h -- C ABI of libmmw.so: the B200-native (sm_100a) implementation of the per-frame
 * radar perception path of AsteriosPar/mmWave_MSc, batched over S independent scenes.
 *
 * The reference has no FFI: its boundary for this path is the Python module API of
 * src/Utils.py and src/Tracking.py.  Every entry point below names the reference
 * interface it replaces (paths relative to the reference's src/).  The Python host layer
 * in mmwave_msc_b200/ binds these with ctypes (mmwave_msc_b200/_lib.py) and mirrors the
 * reference's names on top (mmwave_msc_b200/Tracking.py, Utils.py).
 *
 * Conventions: extern "C"; plain pointers and sizes; no exceptions cross the boundary;
 * every function returns MMW_OK (0) or a negative mmw_status; mmw_last_error() gives the
 * message of the last failure on the calling thread.  The caller owns every buffer it
 * passes in; the context owns all device memory and one CUDA stream.  A context is not
 * thread-safe; distinct contexts are independent.  There is no CPU fallback: without a
 * CUDA device mmw_create fails with MMW_ERR_CUDA.
 */
#ifndef MMW_H
#define MMW_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 7: per-scene export / import (mmw_scene_blob_header, mmw_export_scenes, mmw_import_scenes) (6: mmw_step_packets and
 * mmw_scene_sensor::num_doppler_bins; 5: per-scene sensor table and mmw_reset_scenes).  The state blob and the scene
 * blob carry this number, so blobs written by another version are refused by mmw_state_restore and mmw_import_scenes. */
#define MMW_ABI_VERSION 7

typedef enum mmw_status {
    MMW_OK = 0,
    MMW_ERR_INVALID = -1,      /* bad argument / configuration */
    MMW_ERR_CUDA = -2,         /* CUDA runtime error (message in mmw_last_error) */
    MMW_ERR_CAPACITY = -3,     /* batch larger than the capacity given to mmw_create */
    MMW_ERR_STATE = -4         /* call order (e.g. pose requested before weights were loaded) */
} mmw_status;

/* Mirror of the reference's constants.py (file:line = constants.py).  s_height, s_tilt_deg, z_max, xyz_q_format and
 * doppler_res are the defaults of every scene's entry in the sensor table (mmw_scene_sensor). */
typedef struct mmw_config {
    double s_height;               /* S_HEIGHT :41 */
    double s_tilt_deg;             /* S_TILT :42 */
    double z_max;                  /* scene bound on z', Utils.py:424 (2.5) */
    int32_t frames_batch;          /* FB_FRAMES_BATCH :66; rings hold frames_batch+1 frames (1..3) */
    int32_t db_min_samples;        /* DB_MIN_SAMPLES_MIN :73 */
    double db_z_weight;            /* DB_Z_WEIGHT :70 */
    double db_range_weight;        /* DB_RANGE_WEIGHT :71 */
    double db_eps;                 /* DB_EPS :72 */
    int32_t tr_max_tracks;         /* TR_MAX_TRACKS :85 (only gates whether DBSCAN runs, Tracking.py:693-696) */
    int32_t kf_enable_est;         /* KF_ENABLE_EST :100 */
    double tr_lifetime_dynamic;    /* TR_LIFETIME_DYNAMIC :86 [s] */
    double tr_lifetime_static;     /* TR_LIFETIME_STATIC :87 [s] */
    double tr_vel_thres;           /* TR_VEL_THRES :88 */
    double tr_gate;                /* TR_GATE :89 */
    double kf_q_var;               /* KF_Q_STD :93, passed as a variance (:212) */
    double kf_p_init;              /* KF_P_INIT :96 */
    double kf_group_disp_init;     /* KF_GROUP_DISP_EST_INIT :97 */
    double kf_a_n;                 /* KF_A_N :101 */
    double kf_a_spr;               /* KF_A_SPR :104 */
    double kf_spread_lim[6];       /* KF_SPREAD_LIM :103 */
    int32_t kf_est_pointnum;       /* KF_EST_POINTNUM :102 */
    int32_t xyz_q_format;          /* Q format of int16 point rows (MMW_STEP_INPUT_I16): metres = value / 2^Q; the
                                      xWR14xx demo reports it per frame (ReadDataIWR1443.py:126-128), usually 9 */
    double intensity_mu;           /* INTENSITY_MU :108 */
    double intensity_std;          /* INTENSITY_STD :109 */
    double x_nudge_thres;          /* 0.6, Tracking.py:397 */
    double x_nudge_gain;           /* 0.4, Tracking.py:398 */
    float default_posture[57];     /* MODEL_DEFAULT_POSTURE :112-172 */
    float reserved1;
    /* smart-window projection (the step right after the path: Utils.py:180-219, Visualizer.py:14-29) */
    double m_x, m_y, m_z;          /* M_X, M_Y, M_Z :31-33: the sensitive object behind the window */
    double fade_size_max;          /* V_SCREEN_FADE_SIZE_MAX :50 */
    double fade_size_min;          /* V_SCREEN_FADE_SIZE_MIN :51 */
    double fade_weight;            /* V_SCREEN_FADE_WEIGHT :52 */
    /* Unit of the Doppler column of every point row: doppler [m/s] = row[3] * doppler_res, multiplied in float64 on
     * the device.  The sensor reports dopplerIdx (int16) and the reference forms doppler = dopplerIdx *
     * dopplerResolutionMps in float64 (ReadDataIWR1443.py:163-165) -- a value fp32 cannot hold.  With doppler_res =
     * dopplerResolutionMps the rows carry the index (exact in fp32) and the product is the reference's, bit for bit.
     * 1.0 (default; 0 is read as 1.0): rows carry m/s directly (exact for values that are fp32-representable). */
    double doppler_res;
} mmw_config;

/* Fills *cfg with the reference's default constants. */
int mmw_default_config(mmw_config* cfg);

typedef struct mmw_ctx mmw_ctx;

/* Pose network variants (train.py). */
#define MMW_POSE_2D 0   /* define_CNN    train.py:33-68  : (8,8,5)   -> 57, used when frames_batch == 0 */
#define MMW_POSE_3D 1   /* define_CNN_3D train.py:71-106 : (3,8,8,5) -> 57, used when frames_batch == 2 */

/* mmw_step flags */
#define MMW_STEP_POSE          0x1u   /* run estimate_posture after track (offline_main.py:60) */
#define MMW_STEP_DEVICE_INPUT  0x2u   /* pts/offsets/dt are device pointers (already resident in HBM) */
#define MMW_STEP_RECORD_LABELS 0x4u   /* keep the DBSCAN labels of this frame for mmw_get_labels */
#define MMW_STEP_INPUT_I16     0x10u  /* pts is int16 [sum N, 5] = x, y, z (Q format: the scene's xyz_q_format, see
                                         mmw_scene_sensor), dopplerIdx, peakVal -- the sensor's own lattice, 10 bytes per
                                         point instead of 20; converted on the device (exact: x = value / 2^Q, doppler =
                                         dopplerIdx * doppler_res in float64) */
#define MMW_STEP_PIPELINE      0x8u   /* throughput mode (with MMW_STEP_POSE): the pose network of this frame runs on a
                                         second stream and overlaps the tracker of the NEXT frame -- keypoints never feed
                                         back into tracking (Tracking.py:705-734).  The frame's packed result records
                                         are produced as part of the step; fetch them with mmw_read_results_async right
                                         after the call.  Results are bit-identical to the serial mode. */

/* per-scene status bits (mmw_get_status) */
#define MMW_SCENE_POINT_OVERFLOW 0x1u /* a frame had more points than max_points_per_frame (extra points dropped) */
#define MMW_SCENE_TRACK_OVERFLOW 0x2u /* more tracks than the max_tracks capacity (extra clusters dropped) */

/*
 * One context = S independent scenes, each the state that offline_main.py:32-34 creates
 * (TrackBuffer() + the global BatchedData() ring), resident on one GPU.
 *   max_points_per_frame : capacity N_cap of one frame of one scene (e.g. 256; 1024 for the dense cfg)
 *   max_tracks           : capacity T_cap of one scene's effective_tracks list (1..32).  The reference can
 *                          exceed TR_MAX_TRACKS (Tracking.py:585-589, 703), so T_cap should be > tr_max_tracks.
 */
int mmw_create(const mmw_config* cfg, int device, int n_scenes, int max_points_per_frame, int max_tracks,
               mmw_ctx** out);
int mmw_destroy(mmw_ctx* ctx);
const char* mmw_last_error(void);
int mmw_abi_version(void);

/* Resets every scene to the state of a fresh TrackBuffer() + BatchedData() (Tracking.py:504-511, 38-41).  The sensor
 * table (mmw_scene_sensor) is configuration and stays as it is. */
int mmw_reset(mmw_ctx* ctx);

/* Changes mmw_config::doppler_res of a live context, the context's unit, and sets it as every scene's doppler_res
 * (mmw_get_scene_sensors shows the result).  Takes effect with the next call; rows already in the rings are re-read in
 * the new unit, so change it only while they hold none -- e.g. before the first frame. */
int mmw_set_doppler_resolution(mmw_ctx* ctx, double doppler_res);

/* ---- per-scene sensor table ----
 * Each scene is one sensor installation or one recorded experiment, with its own mounting and radar profile.
 * mmw_create fills every scene's entry from the mmw_config; a context that never changes the table behaves as if it
 * had none.  A change takes effect with the next mmw_step, mmw_run_frames*, mmw_estimate_posture,
 * mmw_pose_features_only or mmw_export_track0: it is queued on the context's stream behind all work already queued
 * there.  Rings store raw sensor rows and world coordinates are recomputed from them, so the rows already in a scene's
 * rings are re-read under the new parameters: change a scene's entry before its first frame, or together with
 * mmw_reset_scenes.  The table is not part of the state blob (it is configuration, like mmw_config and the pose
 * weights): a restored context continues with whatever table it has.  The stateless stage entry points
 * (mmw_preprocess, mmw_dbscan) and mmw_decode_tlv keep using the values of the mmw_config; mmw_step_packets decodes each
 * scene's packet with its own num_doppler_bins. */
typedef struct mmw_scene_sensor {
    double s_height;               /* S_HEIGHT constants.py:41 */
    double s_tilt_deg;             /* S_TILT constants.py:42 */
    double z_max;                  /* scene bound on z', Utils.py:424 */
    double doppler_res;            /* unit of the Doppler column, as mmw_config::doppler_res (must be > 0 here) */
    int32_t xyz_q_format;          /* Q format of int16 rows (MMW_STEP_INPUT_I16), 0..15 */
    int32_t num_doppler_bins;      /* the radar profile's numDopplerBins (ReadDataIWR1443.py:167-175), >= 0; only
                                      mmw_step_packets reads it.  0 (what mmw_create sets) = not set */
} mmw_scene_sensor;

/* Sets the entries of scenes first_scene .. first_scene + n - 1 from params[0 .. n-1].  All or nothing: a range out of
 * bounds, a NULL pointer, a non-finite value, doppler_res <= 0, a Q format outside 0..15 or num_doppler_bins < 0 give
 * MMW_ERR_INVALID and change no entry. */
int mmw_set_scene_sensors(mmw_ctx* ctx, int first_scene, int n, const mmw_scene_sensor* params);
/* Reads the entries of scenes first_scene .. first_scene + n - 1 into out[0 .. n-1]. */
int mmw_get_scene_sensors(mmw_ctx* ctx, int first_scene, int n, mmw_scene_sensor* out);

/* mmw_reset restricted to the n listed scenes (e.g. a sensor slot handed to a new sensor): their scene record, track
 * records, ring histograms, per-scene counters of the last step and pose-row count are cleared, so they continue like
 * fresh scenes (track ids restart at 0).  Other scenes, the sensor table, the accumulated counters and results already
 * packed for earlier frames are left alone.  Duplicate or out-of-range indices give MMW_ERR_INVALID and reset nothing. */
int mmw_reset_scenes(mmw_ctx* ctx, const int32_t* scenes, int n);

/* Checkpoint / resume of the tracker state of all scenes (track records, rings, keypoints, id counters): what a
 * replay needs to continue bit-identically in this or another context created with the same n_scenes,
 * max_points_per_frame, max_tracks and frames_batch (e.g. on another GPU).  mmw_state_size() = bytes of the blob;
 * dump / restore take a HOST buffer of at least that size and are synchronous.  The reference has no equivalent
 * (its state lives in Python objects for the length of the process); pose weights and the sensor table are not part
 * of the blob, and a blob of another ABI version is refused. */
size_t mmw_state_size(mmw_ctx* ctx);
int mmw_state_dump(mmw_ctx* ctx, void* host_blob, size_t bytes);
int mmw_state_restore(mmw_ctx* ctx, const void* host_blob, size_t bytes);

/* ---- per-scene export / import: live scenes move between slots, contexts and GPUs ----
 * A scene blob holds the tracker state of n listed scenes of one context -- each scene's slice of what the state blob
 * holds (scene record, track records, keypoints, track rings, unassigned ring, ring histograms, pose-row count) --
 * together with each scene's sensor-table entry: the rings hold raw sensor rows, which are re-read under the entry of
 * the slot they sit in.  Layout: this 64-byte header, the n source scene indices (int32, padded to 16 bytes), then n
 * records of record_bytes each, in list order.  The record's layout is private to the library and versioned by
 * MMW_ABI_VERSION.  Not carried: the outputs of the scene's last frame (point associations, labels, pose rows, packed
 * records), the accumulated counters, and the mmw_config (the tracker constants are the destination's). */
#define MMW_SCENE_BLOB_MAGIC 0x4d4d574du   /* "MMWM"; the state blob's is "MMWS" */
typedef struct mmw_scene_blob_header {
    uint32_t magic;                /* MMW_SCENE_BLOB_MAGIC */
    uint32_t abi_version;          /* MMW_ABI_VERSION of the library that wrote it */
    int32_t n;                     /* scenes in the blob */
    int32_t max_points_per_frame;  /* shape of the context it was exported from: an import needs the same values */
    int32_t max_tracks;
    int32_t frames_batch;
    uint64_t record_bytes;         /* bytes of one scene record (a multiple of 16) */
    uint64_t total_bytes;          /* bytes of the whole blob: mmw_scene_state_size(ctx, n) */
    uint32_t reserved[6];          /* 0 */
} mmw_scene_blob_header;

/* Bytes of a scene blob of n scenes of this context's shape (0 for a NULL ctx or n < 0). */
size_t mmw_scene_state_size(mmw_ctx* ctx, int n);
/* Writes the scenes scenes[0 .. n-1] into host_blob (at least mmw_scene_state_size(ctx, n) bytes, pageable or pinned)
 * and leaves them unchanged: moving a scene is export, import, and mmw_reset_scenes on the source if its slot is to be
 * reused.  Synchronous: waits for the work queued so far, the throughput mode's pose network included.  Errors, with
 * nothing queued: MMW_ERR_INVALID for a NULL pointer, n < 0, or an index out of range or listed twice;
 * MMW_ERR_CAPACITY when bytes is too small.  n = 0 writes a header only. */
int mmw_export_scenes(mmw_ctx* ctx, const int32_t* scenes, int n, void* host_blob, size_t bytes);
/* Puts record i of a scene blob into slot scenes[i] of this context, sensor-table entry included; n must equal the
 * blob's n.  The header (magic, ABI version, shape, sizes), the destination indices and every record field the kernels
 * use as an index or a count are checked on the host first: a failure gives MMW_ERR_INVALID and changes nothing.
 * The slots' per-scene counters of the last step are cleared, as mmw_reset_scenes clears them; their tracks continue
 * where the source's left off (track ids included).  Synchronous, queued behind all work already queued.  n = 0 checks
 * the header and does nothing. */
int mmw_import_scenes(mmw_ctx* ctx, const int32_t* scenes, int n, const void* host_blob, size_t bytes);

/*
 * Loads the keypoint regressor's weights (replaces keras load_model, offline_main.py:33).
 * blob = concatenation of Keras model.get_weights() flattened, fp32 (see mmwave_msc_b200/pose_weights.py).
 */
int mmw_load_pose_weights(mmw_ctx* ctx, int variant, const float* blob, size_t n_floats);

/*
 * One radar frame for every scene: the loop body of offline_main.py:45-60 --
 *   Utils.normalize_data (Utils.py:342-434), TrackBuffer.track (Tracking.py:664-703) and, with
 *   MMW_STEP_POSE, TrackBuffer.estimate_posture (Tracking.py:705-734).
 *   pts     [sum N, 5] fp32 rows x, y, z, doppler, peakVal in the sensor frame (detObj of ReadDataIWR1443.py)
 *   offsets [S+1]      int32 row offsets of each scene's points (ragged batch)
 *   dt      [S]        fp64 seconds since the scene's previous frame (trackbuffer.dt, offline_main.py:45-49)
 * Scenes whose frame is empty after the scene-bounds filter are skipped entirely, as offline_main.py:55 does.
 * Asynchronous on the context's stream unless the inputs are pageable host memory.
 * The flags are checked before the inputs, and a refused call queues nothing.
 */
int mmw_step(mmw_ctx* ctx, const float* pts, const int32_t* offsets, const double* dt, uint32_t flags);

/* TrackBuffer.estimate_posture (Tracking.py:705-734) alone, on the current state of every scene whose last
 * frame ran: feature maps (relative_coordinates + format_single_frame, Utils.py:437-520) + the CNN. */
int mmw_estimate_posture(mmw_ctx* ctx);

/* Builds only the pose rows / feature maps of mmw_estimate_posture (readable with mmw_get_pose_rows) so that a
 * caller-supplied model object can do the inference (Tracking.py:732), and stores its answer for one track. */
int mmw_pose_features_only(mmw_ctx* ctx);
int mmw_set_keypoints(mmw_ctx* ctx, int scene, int track_index, const float* keypoints57);

/* Blocks until all work queued on the context's stream has finished. */
int mmw_sync(mmw_ctx* ctx);
/* The context's cudaStream_t (so a host framework can time it with events / order copies after it). */
void* mmw_stream(mmw_ctx* ctx);

/* One element of effective_tracks (Tracking.py ClusterTrack/KalmanState/PointCluster attributes). */
typedef struct mmw_track_out {
    int32_t id;                /* value of next_track_id when the track was spawned (Tracking.py:587-588) */
    int32_t point_num;         /* cluster.point_num of the last associated cloud */
    int32_t is_static;         /* cluster.status == STATIC (Tracking.py:132-136) */
    int32_t ring_frames;       /* len(track.batch.buffer) */
    int32_t ring_counts[3];    /* points kept per ring frame, oldest first (at most 64 each are stored) */
    int32_t reserved;
    double lifetime;           /* seconds since the last association (Tracking.py:400-407) */
    double n_est;              /* N_est */
    double x[9];               /* state.x */
    double P[81];              /* state.P row-major */
    double spread_est[6];
    double group_disp_est[36];
    double centroid[6];
    double min_vals[6];
    double max_vals[6];
    float keypoints[57];       /* [x0..x18 | y0..y18 | z0..z18] (train.py:169-177) */
    float reserved2;
} mmw_track_out;

/*
 * Readback (host buffers).  tracks: [S * max_tracks] entries, scene s at tracks[s*max_tracks ..], in
 * effective_tracks list order; n_tracks: [S].  Either pointer may be NULL.
 */
int mmw_get_tracks(mmw_ctx* ctx, mmw_track_out* tracks, int32_t* n_tracks);

/* Compact per-scene summary for the hot loop's result read: n_tracks [S], next_track_id [S],
 * M (points that survived the scene-bounds filter in the last frame) [S].  Any pointer may be NULL. */
int mmw_get_scene_summary(mmw_ctx* ctx, int32_t* n_tracks, int32_t* next_track_id, int32_t* last_M);

/* Per-point association of the last frame, the return value of TrackBuffer._calc_dist_fun
 * (Tracking.py:530-574): assoc[offsets[s] + m] for m < M_s is the index in the pre-maintenance track list,
 * -1 = unassigned (None).  Entries m >= M_s are -2.  assoc: [sum N] int32. */
int mmw_get_point_assoc(mmw_ctx* ctx, int32_t* assoc, size_t n);

/* DBSCAN labels of the last frame stepped with MMW_STEP_RECORD_LABELS: labels [S * 3 * max_points] int32
 * (scene s at s*3*max_points, fused ring order oldest frame first, -1 noise); n_fused [S] = number of fused
 * points clustered, or -1 when DBSCAN did not run for that scene (Tracking.py:693-697). */
int mmw_get_labels(mmw_ctx* ctx, int32_t* labels, int32_t* n_fused);

/* Per-scene overflow bits since creation/reset. */
int mmw_get_status(mmw_ctx* ctx, uint32_t* flags);

/* Sizes of the global unassigned ring (batch.buffer of offline_main.py:34): counts [S*3] oldest first,
 * -1 for absent frames. */
int mmw_get_ring_counts(mmw_ctx* ctx, int32_t* counts);

/* BatchedData.pop_frame / clear on the global ring of one scene (preprocessing.py:263-264, Tracking.py:53-71). */
int mmw_ring_pop(mmw_ctx* ctx, int scene);
int mmw_ring_clear(mmw_ctx* ctx, int scene);

/* Pose input/output of the last MMW_STEP_POSE frame: number of track rows, their (scene, list index) and the
 * feature maps handed to the network, fp32 [(frames_batch+1) * 64 * 5] per row (format_single_frame,
 * Utils.py:468-520).  feats/scene_idx/track_idx may be NULL; *n_rows is always written. */
int mmw_get_pose_rows(mmw_ctx* ctx, int32_t* n_rows, int32_t* scene_idx, int32_t* track_idx, float* feats,
                      size_t feats_capacity_floats);

/* ---- stage-level entry points (stateless; host buffers; used by the known-answer tests) ---- */

/* Utils.normalize_data (Utils.py:342-434) on a ragged batch: world [sum N, 8] fp64 rows
 * x,y,z,vx,vy,vz,doppler,peakVal for every input point and keep [sum N] (1 = inside the scene bounds). */
int mmw_preprocess(mmw_ctx* ctx, const float* pts, size_t n_points, double* world, uint8_t* keep);

/* Utils.apply_DBscan (Utils.py:250-291) with exact epsilon-neighbourhoods on a ragged batch of clouds:
 * xyz [sum B, 3] fp64, offsets [C+1]; labels [sum B] int32 with sklearn's numbering (-1 noise).
 * Each cloud may have at most 3*max_points points.  eps <= 0 / min_samples <= 0 select the config values. */
int mmw_dbscan(mmw_ctx* ctx, const double* xyz, const int32_t* offsets, int n_clouds, double eps, int min_samples,
               int32_t* labels);

/* filterpy KalmanFilter.predict as ClusterTrack.predict_state calls it (Tracking.py:372-385):
 * x [n,9], P [n,81] updated in place with F(dt[i]), Q(dt[i]) of constants.py:195-215. */
int mmw_kalman_predict(mmw_ctx* ctx, double* x, double* P, const double* dt, int n);

/* filterpy KalmanFilter.update (Joseph form) as ClusterTrack.update_state calls it (Tracking.py:387-398),
 * including the x[0] nudge: z [n,6], R [n,36], lifetime_is_zero [n]; x, P updated in place. */
int mmw_kalman_update(mmw_ctx* ctx, double* x, double* P, const double* z, const double* R,
                      const uint8_t* lifetime_is_zero, int n);

/* Gate scores of TrackBuffer._calc_dist_fun (Tracking.py:545-572) for one scene: points [M,6] fp64,
 * tracks given by hx [T,6] and C [T,36]; d2 [M,T] fp64 and assoc [M] int32 out. */
int mmw_gate(mmw_ctx* ctx, const double* points, int M, const double* hx, const double* C, int T, double* d2,
             int32_t* assoc);

/* Keras model.predict (Tracking.py:732): feats [n, (frames_batch+1)*64*5] fp32 -> keypoints [n,57] fp32. */
int mmw_pose(mmw_ctx* ctx, const float* feats, int n, float* keypoints);

/* ---- sensor wire format (SURVEY 8(f) row 4) ---- */

/* Decodes n framed xWR14xx UART packets (each starts with the magic word 02 01 04 03 06 05 08 07) into the ragged
 * fp32 point batch mmw_step takes: what ReadIWR14xx.read (ReadDataIWR1443.py:88-201) extracts from one packet --
 * header, the first TLV if numDetectedObj > 0 and its type is 1 (detected points), objects as six little-endian
 * 16-bit two's-complement words (rangeIdx, dopplerIdx, peakVal, x, y, z), the dopplerIdx correction of :167-175 with
 * the int16 semantics of the reference's numpy 1.26, x y z / 2^xyzQFormat, doppler = dopplerIdx * doppler_res.
 * Finding the packets in a byte stream (magic-word search, waiting for totalPacketLen bytes) stays with the caller.
 *   packets, packet_offsets[n+1]  concatenated packet bytes and their boundaries (host)
 *   points [max_points_total][5]  x y z doppler peakVal (host); point_offsets[n+1]; frame_numbers[n];
 *   data_ok[n] = the reference's dataOK (0: no object, other TLV type, truncated or bad magic -> no points)
 * Pinned to the reference's own ReadIWR14xx.read() run under a numpy-1.x int16 casting shim (27 packets,
 * tests/golden/tlv/reference_tlv.npz; DESIGN.md section 8).  Synchronous. */
int mmw_decode_tlv(mmw_ctx* ctx, const uint8_t* packets, const int64_t* packet_offsets, int n_packets,
                   double num_doppler_bins, double doppler_res, float* points, size_t max_points_total,
                   int32_t* point_offsets, int32_t* frame_numbers, int32_t* data_ok);

/* One radar frame for every scene straight from its sensor's packet: the online loop's ReadIWR14xx.read()
 * (ReadDataIWR1443.py:88-201) followed by mmw_step, with each scene's own radar profile.
 *   packets, packet_offsets[S+1]  host; scene s's packet is bytes [packet_offsets[s], packet_offsets[s+1]): one framed
 *                                 packet as mmw_decode_tlv takes it, or an empty range for no packet.  packet_offsets[0]
 *                                 must be 0.
 *   dt [S]                        host, as for mmw_step
 *   frame_numbers [S], data_ok [S] host or NULL; written before the call returns, as mmw_decode_tlv writes them
 * Each packet is decoded as ReadIWR14xx.read() decodes it: x, y, z = int16 / 2^(the packet's own xyzQFormat), and the
 * Doppler column carries the corrected dopplerIdx, using the scene's num_doppler_bins; the step multiplies it by the
 * scene's doppler_res in float64, so doppler_res must be the profile's dopplerResolutionMps.  A packet with dataOK = 0,
 * or no packet, is an empty frame: the scene is skipped as mmw_step skips it.  The result (overflow bits included) is
 * that of mmw_decode_tlv with doppler_res = mmw_config::doppler_res followed by mmw_step, bit for bit.
 * The headers (a few dozen bytes per packet) are read on the host, to validate the batch and lay out the rows; the
 * bytes go up once, into double-buffered staging on the upload stream, and the objects are decoded on the device into
 * the step's input.  flags: MMW_STEP_POSE, MMW_STEP_PIPELINE and MMW_STEP_RECORD_LABELS as for mmw_step;
 * MMW_STEP_INPUT_I16 and MMW_STEP_DEVICE_INPUT give MMW_ERR_INVALID.  Errors, with nothing queued: MMW_ERR_INVALID for
 * bad offsets or a NULL pointer; MMW_ERR_CAPACITY for more decoded points than n_scenes * max_points_per_frame;
 * MMW_ERR_STATE for a scene whose packet yields objects while its num_doppler_bins is 0.  Host buffers as for mmw_step:
 * keep them unchanged until the next-but-one step; asynchronous for pinned memory.  mmw_get_point_assoc,
 * mmw_get_labels, mmw_read_results_async and the throughput mode work after it as after mmw_step. */
int mmw_step_packets(mmw_ctx* ctx, const uint8_t* packets, const int64_t* packet_offsets, const double* dt, uint32_t flags,
                     int32_t* frame_numbers, int32_t* data_ok);

/* ---- dataset-builder mode (SURVEY 8(f) row 3) ---- */

/* What preprocessing.preprocess_dataset (preprocessing.py:185-216) writes after a frame, for every scene at once:
 * valid[s] = 1 iff the scene's last frame ran track(), track 0 exists, was associated in that frame (lifetime == 0)
 * and has points in its ring; then rows[s] is the (192, 5) float64 block of
 * Utils.format_batched_frames(Utils.relative_coordinates(ring frames, centroid)) (Utils.py:523-548, 437-465): ring
 * frames newest first, [x - cx, y - cy, z, doppler, peakVal], first 64 rows per frame, zero padded, unsorted; and
 * centroid[s] = track 0's cluster centroid[:2] (preprocessing.py:209-213).  rows of invalid scenes are zero.
 * Host pointers: rows [S][192][5], valid [S], centroid [S][2] (may be NULL).  Synchronous. */
int mmw_export_track0(mmw_ctx* ctx, double* rows, int32_t* valid, double* centroid);

/* ---- device-side views for a host framework that owns the stream (bench / torch.distributed gather) ---- */

/* Packs the per-scene results of the last frame into a caller-provided DEVICE buffer of
 * S * max_tracks * MMW_RESULT_FLOATS fp32, ready to be all-gathered across ranks.  Record layout:
 *   [0] id (-1 = no track)  [1] n_tracks of the scene  [2..10] state.x  [11..67] keypoints
 *   [68] [69] centre (x, z) of the track's fade square on the smart window = calc_projection_points(
 *        x[0] + kp[3], x[1] + kp[41], kp[22])  (Visualizer.py:16-20, Utils.py:180-219)
 *   [70] side of the fade square (Visualizer.py:21-28)   [71] 0
 * Asynchronous on the context's stream. */
#define MMW_RESULT_FLOATS 72
int mmw_pack_results(mmw_ctx* ctx, float* device_out);

/* The one collective of the path (SURVEY 8(b), 8(e)): scenes are sharded over the GPUs of a box with no traffic in
 * the hot loop; the packed result records of all ranks are gathered with ONE ncclAllGather over NVLink/NVSwitch.
 *   nccl_comm      : an ncclComm_t whose ranks each own one context of the same n_scenes / max_tracks
 *   device_out_all : DEVICE buffer of nranks * S * max_tracks * MMW_RESULT_FLOATS fp32; rank r's records land in block
 *                    r.  This rank's records are packed straight into its own block (no staging copy) and the
 *                    all-gather runs in place on the context's stream; asynchronous.
 * libnccl.so.2 is bound at run time (dlopen: the copy the process already loaded, e.g. PyTorch's); the call fails
 * with MMW_ERR_STATE when there is none.  mmw_nccl_* are conveniences for a host without an NCCL binding of its own:
 * rank 0 calls mmw_nccl_unique_id (128 bytes), ships the bytes to the others by any means, every rank calls
 * mmw_nccl_comm_init. */
int mmw_gather_nccl(mmw_ctx* ctx, void* nccl_comm, int nranks, float* device_out_all);
int mmw_nccl_unique_id(void* id128);
int mmw_nccl_comm_init(mmw_ctx* ctx, const void* id128, int nranks, int rank, void** nccl_comm_out);
int mmw_nccl_comm_destroy(void* nccl_comm);

/* Pipelined result read-back for the hot loop: packs the results of the frames queued so far (same layout as
 * mmw_pack_results) and downloads them into host_out (pinned memory recommended; S * max_tracks *
 * MMW_RESULT_FLOATS fp32) on a side stream, without blocking the host.  *slot receives the id (0/1) to pass to
 * mmw_wait_results, which blocks until that download has finished.  Together with mmw_step on pinned host inputs
 * (uploaded on another side stream into double-buffered staging) the upload of frame k+1, the kernels of frame k
 * and the download of frame k-1 overlap.  Host input buffers must stay unchanged until the next-but-one
 * mmw_step or mmw_sync. */
int mmw_read_results_async(mmw_ctx* ctx, float* host_out, int* slot);
int mmw_wait_results(mmw_ctx* ctx, int slot);

/* The replay loop of offline_main.py:40-62 for all scenes of the context, n_frames frames back to back from HOST
 * buffers (pinned memory recommended), in C: frame f takes its rows at pts + frame_row_offsets[f] rows (fp32 rows, or
 * int16 rows with MMW_STEP_INPUT_I16), its own CSR offsets at offsets + f * (S + 1) (each starting at 0) and dt + f * S,
 * and leaves its packed result records (layout of mmw_pack_results) at results + f * S * max_tracks *
 * MMW_RESULT_FLOATS.  flags as for mmw_step (MMW_STEP_POSE | MMW_STEP_PIPELINE for the throughput mode).  The upload
 * of frame f+1, the kernels of frame f and the download of frame f-1 overlap; returns when every frame's results
 * are in host memory. */
int mmw_run_frames(mmw_ctx* ctx, int n_frames, const void* pts, const int64_t* frame_row_offsets, const int32_t* offsets,
                   const double* dt, float* results, uint32_t flags);

/* mmw_run_frames that sends back only the records of LIVE tracks (a scene holds ~2 of its max_tracks slots: a quarter of
 * the bytes).  Frame f leaves n_records[f] records at results + f * S * max_tracks * MMW_RESULT_FLOATS (the same frame
 * stride as mmw_run_frames, only the head of each frame's block is written), in (scene, list index) order; field [71]
 * of a record is its scene index, field [1] the scene's track count, the other fields as in mmw_pack_results.  Scenes
 * without tracks leave no record.  The records are written by a kernel straight into the host buffer, so `results`
 * and `n_records` must be pinned, device-mapped host memory (cudaHostAlloc / cudaHostRegister, e.g. torch
 * pin_memory()); MMW_ERR_INVALID otherwise. */
int mmw_run_frames_compact(mmw_ctx* ctx, int n_frames, const void* pts, const int64_t* frame_row_offsets,
                           const int32_t* offsets, const double* dt, float* results, int32_t* n_records, uint32_t flags);

/* Counters accumulated on the device since the last call (algorithmic-bytes bookkeeping, SURVEY 8(d)):
 * out[0]=frames stepped (scene-frames that ran), [1]=sum N, [2]=sum M, [3]=sum U (unassigned pushed),
 * [4]=sum fused points clustered, [5]=sum tracks after the frame, [6]=sum min(A_j,64) ring rows written,
 * [7]=pose rows. */
int mmw_get_counters(mmw_ctx* ctx, uint64_t out[8], int reset);

/* Selects the kernel used for the pose network's dense contraction: 1 = tcgen05 tensor-core path (default),
 * 0 = CUDA-core fp32 path (kept for numerics comparison). */
int mmw_set_dense_path(mmw_ctx* ctx, int use_tensor_cores);

/* Test hook: intermediates of the last pose-network run on the context's main stream (mmw_pose, or a serial
 * mmw_step / mmw_estimate_posture with MMW_STEP_POSE), rows in that run's order, positions in Keras order (d, h, w, c):
 *   layer 0: network input as split for the tensor cores    [n][D*64][5]
 *   layer 1: conv 1 after ReLU                               [n][D*64][16]
 *   layer 2: conv 2 after ReLU and BN 1 (the Flatten order)  [n][D*64*32]
 *   layer 3: dense 1 after ReLU and BN 2                     [n][H]
 * Tensor-core path: two uint16 planes of n * (values per row) each, the raw bf16 bits of hi, then of lo.  CUDA-core
 * path: fp32, layers 2 and 3 only (MMW_ERR_INVALID for 0 and 1).  *n_rows = n of that run; host_out may be NULL to
 * ask for n only, otherwise it must hold the whole layer (MMW_ERR_CAPACITY).  MMW_ERR_STATE: no weights loaded, no run
 * since they were loaded (or since mmw_reset / mmw_pose_features_only), or the last run was in throughput mode (its
 * intermediates belong to a frame that may still be in flight).  Synchronous. */
int mmw_pose_intermediate(mmw_ctx* ctx, int layer, int* n_rows, void* host_out, size_t bytes);

/* Per-kernel device time: while enabled, every launch of mmw_step / mmw_step_packets is bracketed by CUDA events on the context's
 * stream.  mmw_get_kernel_ms returns the accumulated milliseconds and launch counts per kernel class. */
#define MMW_K_STEP 0           /* fused tracker step (normalize + track) */
#define MMW_K_POSE_INDEX 1     /* pose row compaction */
#define MMW_K_POSE_FEATURES 2  /* relative_coordinates + format_single_frame */
#define MMW_K_CONV 3           /* conv1 + conv2 + BatchNorm */
#define MMW_K_FC1 4            /* dense 1 (+ operand split when the tensor-core path is on) */
#define MMW_K_FC2 5            /* dense 2 */
#define MMW_K_DBSCAN_BIG 6     /* union / border / spawn of the few scenes per frame in which clusters form */
#define MMW_K_PACKETS 7        /* decode of the packets of mmw_step_packets into the step's input */
#define MMW_N_KERNELS 8
int mmw_profile(mmw_ctx* ctx, int enable);
int mmw_get_kernel_ms(mmw_ctx* ctx, double* total_ms /*[MMW_N_KERNELS]*/, uint64_t* calls /*[MMW_N_KERNELS]*/);

/* Debug: per-phase SM-cycle accounting inside the fused step kernel (thread 0 of every CTA).  Returns the
 * cycles accumulated since the last call in out16 (may be NULL) and switches the accounting on/off. */
int mmw_phase_clocks(mmw_ctx* ctx, int enable, uint64_t* out16);
/* Debug: SM cycles the step kernel spent on each scene in the last frame stepped with the accounting on. */
int mmw_scene_cycles(mmw_ctx* ctx, uint64_t* out /*[3*S]: cycles, then start and end %globaltimer ns per scene*/);

/* Debug: cycles of dbscan_big_kernel (thread 0 of each CTA, summed over the deferred scenes) since the last call, while
 * mmw_phase_clocks is on: [0] ring load [1] labels+spawn+write-back [2] scenes [3] adjacency + counts [5] components
 * [6] border points [7] fused points; the rest is reserved.  out16: 16 values. */
int mmw_dbscan_big_clocks(mmw_ctx* ctx, uint64_t* out16);

/* Number of kernels this library launched since creation (bench.py's gpu_launches). */
uint64_t mmw_launch_count(mmw_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* MMW_H */
