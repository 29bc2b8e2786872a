// Internal device-side data model of libmmw (see DESIGN.md "Data layout in HBM").
#pragma once
#include <utility>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/mmw.h"

namespace mmw {

constexpr int kRing = 3;          // max frames in a ring: FB_FRAMES_BATCH + 1 <= 3 (constants.py:66)
constexpr int kFeatPts = 64;      // points kept per track ring frame (format_single_frame, Utils.py:505-510)
constexpr int kRawCols = 5;       // x, y, z, doppler, peakVal (sensor frame, fp32)
constexpr int kKp = 57;           // 19 joints x 3
constexpr int kHistBytes = 272;   // per ring frame: 256 cell counts of the grid screen (uint8, saturating) + flag + pad
constexpr int kStepThreads = 128;    // threads per scene CTA of the tracker step
constexpr int kStepWarps = kStepThreads / 32;
constexpr int kMaxTcap = 32;

// One scene's sensor mounting and radar profile (mmw_scene_sensor) as the kernels use it: one record per scene in
// HBM (mmw_ctx::d_sensors), read by every kernel that turns raw rows into world coordinates.
struct SensorRec {
    double cos_t, sin_t, s_height, z_max;
    double doppler_res;        // doppler [m/s] = row[3] * doppler_res (float64 product, ReadDataIWR1443.py:163-165)
    float xyz_scale;           // 2^-Q of int16 point rows (MMW_STEP_INPUT_I16)
    int32_t pad;
};
static_assert(sizeof(SensorRec) == 48, "SensorRec is three 16-byte chunks (moved with one bulk copy)");

// The record read where it is used: volatile loads are not hoisted out of loops, so a kernel at its register limit does
// not keep the values live (and spilled) between uses, which kernel parameters never needed.
__device__ __forceinline__ SensorRec sensor_at_use(const SensorRec& r) {
    const volatile SensorRec& v = r;
    SensorRec o;
    o.cos_t = v.cos_t; o.sin_t = v.sin_t; o.s_height = v.s_height; o.z_max = v.z_max;
    o.doppler_res = v.doppler_res; o.xyz_scale = v.xyz_scale; o.pad = 0;
    return o;
}

// One scene's tracker and DBSCAN constants (mmw_scene_tracker) as the kernels use it, with what is derived from them
// per entry on the host: one record per scene in HBM (mmw_ctx::d_trackers), read by step_kernel and dbscan_big_kernel.
struct TrackerRec {
    double db_z_weight, db_range_weight, db_eps;
    double life_dyn, life_sta, vel_thres, gate;
    double q_var, p_init, g_init, a_n, a_spr;
    double spread_lim[6];
    double nudge_thres, nudge_gain;
    int32_t db_min_samples, tr_max_tracks, enable_est, est_pointnum;
    // grid screen in front of DBSCAN (dbscan.cuh): fixed 16 x 16 cells over world (x, y'), at least one eps reach wide
    // for every pair of points with y' <= grid_ybound; grid_ok = 0: degenerate configuration, the screen always passes
    float grid_inv_h, grid_ybound;
    int32_t grid_ok;
    // fp32 screen of the eps predicate (dbscan.cuh, screen_d): guard band [lo, hi] around eps, and the domain |y'|, |z'|
    // <= rmax in which the band covers the fp32 error (rmax = -1: every pair is decided in float64)
    float screen_lo, screen_hi, screen_rmax;
    int32_t pad[2];
};
static_assert(sizeof(TrackerRec) == 208, "TrackerRec is thirteen 16-byte chunks (moved with one bulk copy)");

// Derived constants handed to kernels by value.
struct DevConfig {
    SensorRec sensor;          // the mmw_config's mounting: the stateless stage entry points use it
    TrackerRec tracker;        // the mmw_config's tracker constants: the stateless stage entry points use them
    double int_mu, int_std;
    int ring_size;
    int ncap, tcap;
};

// One element of a scene's effective_tracks list (ClusterTrack + KalmanState + PointCluster).
// All decision arithmetic of the tracker is float64, like the reference.
struct TrackRec {
    double x[9];
    double P[81];
    double spread[6];
    double G[36];          // group_disp_est
    double centroid[6];
    double minv[6];
    double maxv[6];
    double n_est;
    double lifetime;
    int32_t id;
    int32_t point_num;
    int32_t is_static;
    int32_t slot;          // physical slot of this track's ring / keypoints inside the scene
    int32_t ring_n;        // frames in the track ring
    int32_t ring_head;     // physical index of the oldest frame
    int32_t ring_cnt[kRing];   // stored rows per PHYSICAL frame (<= 64)
    int32_t pad[3];            // record = 1264 bytes = 79 x 16 (moved with 16-byte cp.async)
};
static_assert(sizeof(TrackRec) % 16 == 0, "TrackRec must be a whole number of 16-byte chunks");
constexpr int kTrackWords = sizeof(TrackRec) / 8;

struct SceneRec {
    int32_t n_tracks;
    int32_t next_id;
    int32_t ring_n;            // frames in the global unassigned ring
    int32_t ring_head;         // physical index of the oldest frame
    int32_t ring_cnt[kRing];   // points per PHYSICAL frame
    uint32_t slot_mask;        // physical track slots in use
    uint32_t flags;            // MMW_SCENE_* overflow bits
    int32_t last_M;            // points surviving the bounds filter in the last frame
    int32_t last_ran;          // 1 if the last frame ran track()
    int32_t dbscan_n;          // fused points clustered in the last frame, -1 if DBSCAN did not run
    int32_t pose_base;         // first pose row of this scene in the last pose batch
    int32_t ring_ph_gone;      // 0 while the global ring still holds the deque's initial empty frame (RingBuffer.__init__
                               //   appends init_val, Utils.py:36-50): it is what batch.pop_frame() pops first
    int32_t pad[2];
};
static_assert(sizeof(SceneRec) == 64, "SceneRec is one 64-byte record");

struct StepArgs {
    DevConfig cfg;
    const SensorRec* sensors;  // [S] each scene's mounting and radar profile
    const TrackerRec* trackers;  // [S] each scene's tracker and DBSCAN constants
    const float* pts;          // [sum N, 5] fp32 rows; int16 rows when flags has MMW_STEP_INPUT_I16
    const int32_t* offsets;    // [S+1]
    const double* dt;          // [S]
    TrackRec* tracks;          // [S][tcap]
    SceneRec* scenes;          // [S]
    float* track_ring;         // [S][tcap][kRing][64][5]
    float* uring;              // [S][kRing][ncap][5]
    float* keypoints;          // [S][tcap][57] by physical slot
    const float* default_posture;  // [57]
    int32_t* assoc_out;        // [sum N]
    int32_t* labels_out;       // [S][3*ncap] or nullptr
    unsigned long long* counters;  // [8]
    unsigned long long* phase_cycles;  // [16 + S] or nullptr: cycles per phase of step_kernel, then cycles per scene (debug)
    int32_t* defer_list;       // [S] scenes whose DBSCAN + spawn is left to dbscan_big_kernel, or nullptr
    int32_t* defer_count;      // device counter of defer_list; dbscan_big_kernel's last CTA zeroes it for the next step
    int32_t* defer_done;       // CTAs of dbscan_big_kernel that have finished (ticket for that reset)
    int32_t* defer_hint;       // mapped host word: the work-list length of this step, read by the host (without any
                               //   synchronisation) to size dbscan_big_kernel's grid of the NEXT steps; or nullptr
    int32_t* pose_cnt;         // [S] tracks of the scene if the frame ran track(), else 0: the pose-row scan reads this
    uint8_t* ring_hist;        // [S][kRing][kHistBytes] cell histograms of the global ring's frames, by physical slot
    int32_t* scene_stats;      // [S][8] this frame's N, M, U, Bf (if DBSCAN ran), tracks, ring rows written, ran, 0:
                               //   summed into `counters` by dbscan_big_kernel (one reduction instead of 7 atomics per scene)
    int n_scenes;
    uint32_t flags;
    // Pose rows of the tracks dbscan_big_kernel spawns (fused MMW_STEP_POSE steps, S <= 4096): the feature kernel lays
    // out the rows of the tracks that existed when step_kernel finished and does not wait for dbscan_big_kernel at all;
    // that kernel computes the feature maps of its new tracks itself and appends them behind (nr_extra counts them).
    // nr_extra == nullptr: the feature kernel runs after dbscan_big_kernel and lays out every track.
    float* nr_feats = nullptr;
    void* nr_packed = nullptr;         // __nv_bfloat16 packed conv-1 input, or nullptr
    int32_t *nr_row_scene = nullptr, *nr_row_track = nullptr, *nr_row_slot = nullptr;
    int32_t* nr_extra = nullptr;
    long long pts_row0 = 0;    // row of `pts` at which this frame starts (offsets are relative to it): lets several frames
                               //   share one 16-byte aligned upload (mmw_run_frames)
};

// ---- programmatic dependent launch (PDL) ----------------------------------------------------------------
// The seven kernels of a step run back to back on one stream.  Each is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, does the part of its prologue that needs nothing from its
// predecessor (barrier init, TMEM allocation, shared-memory zero fill, tensor-map prefetch), then
// pdl_wait() -- the predecessor grid has completed and its writes are visible -- and only then
// pdl_launch_dependents(), so that whenever a kernel's CTAs start, the kernel TWO places upstream has completed.
// Launch latency and prologues overlap the predecessor's tail instead of sitting between kernels.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// kernel<<<grid, block, smem, st>>>(args...) with the PDL attribute (and an optional cluster shape)
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              dim3 cluster, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int n = 0;
    if (cluster.x * cluster.y * cluster.z > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = cluster.x; at[n].val.clusterDim.y = cluster.y; at[n].val.clusterDim.z = cluster.z;
        ++n;
    }
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
    cfg.attrs = at; cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// cudaFuncSetAttribute is per device and a process may hold contexts on several GPUs: every launcher keeps what it
// has asked for per device.  smem < 0: only the carve-out preference.
constexpr int kMaxDevices = 64;
inline cudaError_t ensure_smem_attr(const void* fn, int* configured /*[kMaxDevices], zero-initialised*/, int smem) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    const int want = smem < 0 ? 1 : smem;
    if (want > configured[dev]) {
        if (smem >= 0) {
            e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (e != cudaSuccess) return e;
        }
        e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        configured[dev] = want;
    }
    return cudaSuccess;
}

// ---- world-frame point from a raw sensor point (Utils.py:379-420) -----------------------------------
// Written with explicit round-to-nearest multiplies/adds (no FMA contraction) so that the
// scene-bounds predicates and the DBSCAN inputs are bit-identical to the float64 numpy oracle.
__device__ __forceinline__ void world_yz(const SensorRec& c, double y, double z, double& yw, double& zw) {
    yw = __dadd_rn(__dmul_rn(c.cos_t, y), __dmul_rn(-c.sin_t, z));
    zw = __dadd_rn(__dadd_rn(__dmul_rn(c.sin_t, y), __dmul_rn(c.cos_t, z)), c.s_height);
}

// (a + b) mod ring_size for 0 <= a + b < 3 * ring_size (ring positions: ring_size <= kRing): two conditional
// subtractions instead of an integer division by a run-time value.
__device__ __forceinline__ int ring_wrap(int v, int ring_size) {
    v = v >= ring_size ? v - ring_size : v;
    return v >= ring_size ? v - ring_size : v;
}

// num / den, correctly rounded like __ddiv_rn.  A zero numerator over a finite non-zero denominator (Doppler bin 0 on a third of
// the points, the identity columns of a Gauss-Jordan step) sends the whole warp down the slow path of the
// division routine -- ~70 instructions, 13.5 % of the step kernel's instructions in the ncu capture
// (profiles/r01_ncu_full_final3.md) -- so it is answered directly: 0 / den = 0 with the sign of num * den.
__device__ __forceinline__ double div_zero_fast(double num, double den) {
    const bool z = num == 0.0 && den != 0.0 && fabs(den) <= 1.7976931348623157e308;   // 0/0, 0/inf, 0/nan: the real thing
    double nsafe = z ? 1.0 : num;
    // opaque to the compiler: it would otherwise divide `num` itself (the quotient is unused when z) -- and did
    asm("" : "+d"(nsafe));
    const double q = __ddiv_rn(nsafe, den);
    return z ? (den < 0.0 ? -num : num) : q;
}

__device__ __forceinline__ void world_from_raw(const SensorRec& c, float fx, float fy, float fz, float fd,
                                               double w[6]) {
    const double x = fx, y = fy, z = fz, d = __dmul_rn((double)fd, c.doppler_res);
    const double r = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));
    double vx, vy, vz;
    if (r == 0.0) {                       // Utils.py:387-390
        vx = 0.0; vy = d; vz = 0.0;
    } else {                              // Utils.py:400-402: (doppler * coord) / r
        vx = div_zero_fast(__dmul_rn(d, x), r);
        vy = div_zero_fast(__dmul_rn(d, y), r);
        vz = div_zero_fast(__dmul_rn(d, z), r);
    }
    w[0] = x;
    world_yz(c, y, z, w[1], w[2]);
    w[3] = vx;
    w[4] = __dadd_rn(__dmul_rn(c.cos_t, vy), __dmul_rn(-c.sin_t, vz));
    w[5] = __dadd_rn(__dmul_rn(c.sin_t, vy), __dmul_rn(c.cos_t, vz));
}

struct FadeCfg { double m_x, m_y, m_z, smax, smin, weight; };

// calc_projection_points (Utils.py:180-219): where the line from the point to the sensitive object (M_X, M_Y, M_Z)
// crosses the window plane y = 0.
__device__ __forceinline__ void projection_point(const FadeCfg& f, double xo, double yo, double zo, double& xp,
                                                 double& zp) {
    const double xd = xo - f.m_x, yd = yo - f.m_y, zd = zo - f.m_z;
    xp = (xd == 0.0) ? xo : (-f.m_y / (yd / xd)) + f.m_x;
    zp = (zd == 0.0) ? zo : (-f.m_y / (yd / zd)) + f.m_z;
}

// Fade square of a packed result record (calc_fade_square, Visualizer.py:14-29), float64 like the reference: rec[2..10]
// = state x, kp = the track's 57 keypoints; writes rec[68..71].
__device__ __forceinline__ void write_fade_square(const FadeCfg& fade, double x0, double x1, const float* kp, float* rec) {
    double cx, cz;
    projection_point(fade, x0 + (double)kp[3], x1 + (double)kp[41], (double)kp[22], cx, cz);
    const double size = fmax(fade.smin, fmin(fade.smax, fade.smax - (x1 + (double)kp[12]) * fade.weight));
    rec[68] = (float)cx; rec[69] = (float)cz; rec[70] = (float)size; rec[71] = 0.f;
}

// altered_EuclideanDist(p, q) <= eps (Utils.py:242-247, compared as sklearn's radius query does)
__device__ __forceinline__ bool eps_neighbour(const TrackerRec& c, double x1, double y1, double z1, double x2,
                                              double y2, double z2, double eps) {
    const double w = __dsub_rn(1.0, __dmul_rn(__dmul_rn(__dadd_rn(y1, y2), 0.5), c.db_range_weight));
    const double dx = __dsub_rn(x1, x2), dy = __dsub_rn(y1, y2), dz = __dsub_rn(z1, z2);
    const double q = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)),
                               __dmul_rn(c.db_z_weight, __dmul_rn(dz, dz)));
    return __dmul_rn(w, q) <= eps;
}

}  // namespace mmw
