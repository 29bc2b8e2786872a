// C ABI of libmmw.so (include/mmw.h): context management, the per-frame step, readback, and the
// stage-level entry points.  No torch types, no exceptions across the boundary, no CPU fallback.
#include <algorithm>
#include <climits>
#include <dlfcn.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "dbscan.cuh"
#include "linalg.cuh"
#include "mmw_internal.cuh"
#include "pose.cuh"
#include "pose_tc.cuh"

using namespace mmw;

static thread_local std::string g_err;

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(MMW_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));        \
    } while (0)

// mmw_run_frames uploads the inputs of kGroup consecutive frames in ONE copy per array (a 2 MB copy runs at 15 GB/s on a
// link that gives 24 GB/s at 8 MB: per-copy cost, not bandwidth)
constexpr int kGroup = 4;
constexpr size_t kStageSlack = 64;   // the step kernel copies 16-byte aligned windows around a scene's rows

// One slot of the input staging of the host-input entry points (see stage_acquire): the inputs of one step, or of a
// group of up to kGroup frames.
struct StageSlot {
    float* pts = nullptr;            // point rows (fp32, or int16 with MMW_STEP_INPUT_I16) of the step or group
    size_t pts_cap = 0;              //   bytes, kStageSlack included
    int32_t* offsets = nullptr;      // [kGroup][S+1]
    double* dt = nullptr;            // [kGroup][S]
    uint8_t* pk = nullptr;           // mmw_step_packets: [S+1] packet offsets (int64) + packet bytes
    size_t pk_cap = 0;
    cudaEvent_t uploaded = nullptr, free = nullptr;
};

struct mmw_ctx {
    mmw_config cfg;
    DevConfig dc;
    int device = 0, S = 0, ncap = 0, tcap = 0;
    cudaStream_t stream = nullptr;
    // sensor table: each scene's mounting and radar profile as set (host) and as the kernels read it (device, [S])
    std::vector<mmw_scene_sensor> sensors;
    SensorRec* d_sensors = nullptr;
    double* d_doppler_wrap = nullptr; // [S] num_doppler_bins / 2 - 1 of each scene: the Doppler threshold of mmw_step_packets
    // resident state
    TrackRec* d_tracks = nullptr;
    SceneRec* d_scenes = nullptr;
    float* d_track_ring = nullptr;
    float* d_uring = nullptr;
    float* d_keypoints = nullptr;
    float* d_default_posture = nullptr;
    int32_t* d_assoc = nullptr;
    int32_t* d_labels = nullptr;
    unsigned long long* d_counters = nullptr;
    unsigned long long* d_phase = nullptr;
    bool phase_clocks = false;
    uint8_t* d_ring_hist = nullptr;   // [S][kRing][kHistBytes] cell histograms of the global ring's frames (grid screen)
    int32_t* h_defer_hint = nullptr;  // pinned + mapped: work-list length of the last finished step (sizes dbscan_big's grid)
    int32_t* d_defer_hint = nullptr;  //   its device alias
    int32_t* h_rows_hint = nullptr;   // pinned + mapped: pose rows of the last finished feature kernel (tile shape of dense 1)
    int32_t* d_rows_hint = nullptr;
    int32_t* d_scene_stats = nullptr; // [S][8] per-scene counters of the last step (summed on the device)
    int32_t* d_defer = nullptr;      // [2 + S + S]: counter, the work list of dbscan_big_kernel, pose rows per scene, finished-CTA ticket
    bool fold_pose_index = true;     // pose-row scan inside pose_feature_kernel (S <= 4096) instead of pose_index_kernel
    // input staging of the host-input entry points, copied on a side stream (see stage_acquire)
    StageSlot stage[2];
    unsigned stage_idx = 0;          // slots taken so far
    unsigned stage_pending = 0;      // bit k: slot k is released, its free event is still to be recorded
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    // throughput mode (MMW_STEP_PIPELINE): pose network on its own stream, its inputs double-buffered
    cudaStream_t pose_stream = nullptr;
    cudaEvent_t feat_done[2] = {nullptr, nullptr}, packt_done[2] = {nullptr, nullptr}, pose_done[2] = {nullptr, nullptr};
    int32_t *d_row_scene2 = nullptr, *d_row_track2 = nullptr, *d_row_slot2 = nullptr;
    int* d_pose_total2 = nullptr;
    int32_t* d_pose_extra = nullptr; // [2] rows dbscan_big_kernel appended for the tracks it spawned (fused steps), by input buffer
    int rows_buf = 0;                // row maps / pose_total of the last feature launch (0 / 1)
    unsigned pipe_idx = 0;           // pipelined steps so far
    int pipe_r = -1;                 // result buffer the last step filled itself (-1: the last step was serial)
    bool pose_pending = false;       // the pose stream has work the main stream has not waited for
    cudaEvent_t packed[2] = {nullptr, nullptr}, results_done[2] = {nullptr, nullptr};
    float* d_results[2] = {nullptr, nullptr};
    double* d_export = nullptr;      // [S][192*5 + 2] rows + centroid of mmw_export_track0 (allocated on first use)
    int32_t* d_export_valid = nullptr;
    unsigned char* d_move = nullptr; // scene blob of mmw_export_scenes / mmw_import_scenes (grown inside those calls only)
    size_t move_cap = 0;
    unsigned result_idx = 0;
    // pose
    int variant = -1;
    bool has_weights = false;
    int D = 0, Kf = 0, H = 0;
    float* d_blob = nullptr;
    const float *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr, *wd1 = nullptr, *bd1 = nullptr,
                *wd2 = nullptr, *bd2 = nullptr;
    float *d_bn1s = nullptr, *d_bn1t = nullptr, *d_bn2s = nullptr, *d_bn2t = nullptr;
    float* d_feats = nullptr;
    int32_t *d_row_scene = nullptr, *d_row_track = nullptr, *d_row_slot = nullptr;
    int* d_pose_total = nullptr;
    float *d_act2 = nullptr, *d_act3 = nullptr, *d_pose_out = nullptr;
    int pose_cap = 0;
    PoseTc tc;              // tensor-core dense path (pose_tc.cu)
    bool use_tc = true;
    // the last pose-network run, for mmw_pose_intermediate: 0 = none (or its buffers were overwritten since),
    // 1 = serial on the tensor cores, 2 = serial on the CUDA cores, 3 = throughput mode
    int last_pose_run = 0;
    uint64_t launches = 0;
    // per-kernel CUDA-event profiling (mmw_profile)
    bool profiling = false;
    std::vector<std::pair<cudaEvent_t, int>> marks;   // event recorded BEFORE kernel `second` (-1 = end marker)
    double kernel_ms[MMW_N_KERNELS] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint64_t kernel_calls[MMW_N_KERNELS] = {0, 0, 0, 0, 0, 0, 0, 0};
};

// Everything queued so far on both compute streams has completed (the pose stream only runs in throughput mode).
static cudaError_t sync_main(mmw_ctx* x) {
    if (x->pose_pending) {
        cudaError_t e = cudaStreamSynchronize(x->pose_stream);
        if (e != cudaSuccess) return e;
        x->pose_pending = false;
    }
    return cudaStreamSynchronize(x->stream);
}
// Serial-mode work is about to be queued on the main stream: it must come after whatever the pose stream still runs.
static cudaError_t join_pose(mmw_ctx* x) {
    if (!x->pose_pending) return cudaSuccess;
    x->pose_pending = false;
    return cudaStreamWaitEvent(x->stream, x->pose_done[(x->pipe_idx + 1) & 1], 0);     // the last pipelined step's
}

static void prof_mark(mmw_ctx* x, int next_kernel) {
    if (!x->profiling) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, x->stream);
    x->marks.emplace_back(e, next_kernel);
}

// The kernels' form of one sensor-table entry.  Every entry, the context default included, is built here: the transform
// is bit-exact to numpy's only while std::cos / std::sin of deg * (pi / 180) agree with np.cos / np.sin(np.radians(deg)).
static SensorRec sensor_rec(const mmw_scene_sensor& p) {
    SensorRec r{};
    const double ang = p.s_tilt_deg * (M_PI / 180.0);      // numpy.radians
    r.cos_t = std::cos(ang);
    r.sin_t = std::sin(ang);
    r.s_height = p.s_height;
    r.z_max = p.z_max;
    r.doppler_res = p.doppler_res;
    r.xyz_scale = (float)std::ldexp(1.0, -(p.xyz_q_format));
    return r;
}

// Threshold of the dopplerIdx correction of mmw_step_packets (ReadDataIWR1443.py:167-175): the value mmw_decode_tlv
// computes from its num_doppler_bins argument.
static double doppler_wrap(const mmw_scene_sensor& p) { return (double)p.num_doppler_bins / 2 - 1; }

// The sensor-table entry every scene starts with: the mmw_config's values (doppler_res 0 is read as 1.0), no
// num_doppler_bins.
static mmw_scene_sensor config_sensor(const mmw_config& c) {
    mmw_scene_sensor p{};
    p.s_height = c.s_height;
    p.s_tilt_deg = c.s_tilt_deg;
    p.z_max = c.z_max;
    p.doppler_res = c.doppler_res != 0.0 ? c.doppler_res : 1.0;
    p.xyz_q_format = c.xyz_q_format;
    return p;
}

static void fill_devconfig(const mmw_config& c, int ncap, int tcap, DevConfig* d) {
    d->sensor = sensor_rec(config_sensor(c));
    d->db_z_weight = c.db_z_weight;
    d->db_range_weight = c.db_range_weight;
    d->db_eps = c.db_eps;
    d->life_dyn = c.tr_lifetime_dynamic;
    d->life_sta = c.tr_lifetime_static;
    d->vel_thres = c.tr_vel_thres;
    d->gate = c.tr_gate;
    d->q_var = c.kf_q_var;
    d->p_init = c.kf_p_init;
    d->g_init = c.kf_group_disp_init;
    d->a_n = c.kf_a_n;
    d->a_spr = c.kf_a_spr;
    for (int i = 0; i < 6; ++i) d->spread_lim[i] = c.kf_spread_lim[i];
    d->int_mu = c.intensity_mu;
    d->int_std = c.intensity_std;
    d->nudge_thres = c.x_nudge_thres;
    d->nudge_gain = c.x_nudge_gain;
    d->db_min_samples = c.db_min_samples;
    d->ring_size = c.frames_batch + 1;
    d->tr_max_tracks = c.tr_max_tracks;
    d->enable_est = c.kf_enable_est;
    d->est_pointnum = c.kf_est_pointnum;
    d->ncap = ncap;
    d->tcap = tcap;
    grid_screen_config(c.db_eps, c.db_range_weight, c.db_z_weight, c.db_min_samples, &d->grid_inv_h, &d->grid_ybound,
                       &d->grid_ok);
    screen_config(c.db_eps, c.db_range_weight, c.db_z_weight, &d->screen_lo, &d->screen_hi, &d->screen_rmax);
}

static const float kDefaultPosture[57] = {
    0.0000f, -0.0007f, -0.0006f, -0.0038f, -0.1820f, -0.2540f, -0.2579f, 0.1830f, 0.2957f, 0.2940f,
    -0.0805f, -0.1141f, -0.1232f, -0.1358f, 0.0796f, 0.1436f, 0.1558f, 0.1720f, -0.0007f, 0.7699f,
    1.0906f, 1.4020f, 1.5513f, 1.2893f, 1.0360f, 0.7994f, 1.2865f, 1.0483f, 0.8117f, 0.7670f,
    0.3428f, 0.0000f, -0.0746f, 0.7713f, 0.3706f, -0.0128f, -0.0796f, 1.3255f, 0.0752f, 0.0533f,
    0.0203f, 0.0000f, 0.0496f, 0.1350f, 0.1303f, 0.0345f, 0.1277f, 0.1050f, 0.0392f, 0.0533f,
    0.0786f, -0.0056f, 0.0346f, -0.0007f, 0.0683f, -0.0082f, 0.0312f};

extern "C" {

int mmw_abi_version(void) { return MMW_ABI_VERSION; }
const char* mmw_last_error(void) { return g_err.c_str(); }

int mmw_default_config(mmw_config* c) {
    if (!c) return fail(MMW_ERR_INVALID, "cfg is NULL");
    std::memset(c, 0, sizeof(*c));
    c->s_height = 1.8; c->s_tilt_deg = -5; c->z_max = 2.5;
    c->frames_batch = 2; c->db_min_samples = 35;
    c->db_z_weight = 0.4; c->db_range_weight = 0.03; c->db_eps = 0.3;
    c->tr_max_tracks = 4; c->kf_enable_est = 0;
    c->tr_lifetime_dynamic = 3; c->tr_lifetime_static = 7; c->tr_vel_thres = 0.12; c->tr_gate = 4.5;
    c->kf_q_var = 1; c->kf_p_init = 0.1; c->kf_group_disp_init = 0.1; c->kf_a_n = 0.9; c->kf_a_spr = 0.9;
    const double lim[6] = {0.2, 0.2, 2, 1.2, 1.2, 0.2};
    for (int i = 0; i < 6; ++i) c->kf_spread_lim[i] = lim[i];
    c->kf_est_pointnum = 10;
    c->intensity_mu = 27.0187; c->intensity_std = 70.351;
    c->x_nudge_thres = 0.6; c->x_nudge_gain = 0.4;
    std::memcpy(c->default_posture, kDefaultPosture, sizeof(kDefaultPosture));
    c->m_x = 0.32; c->m_y = -0.6; c->m_z = 1.3;
    c->fade_size_max = 0.3; c->fade_size_min = 0.2; c->fade_weight = 0.08;
    c->doppler_res = 1.0;
    c->xyz_q_format = 9;
    return MMW_OK;
}

int mmw_destroy(mmw_ctx* x) {
    if (!x) return MMW_OK;
    cudaSetDevice(x->device);
    if (x->stream) cudaStreamSynchronize(x->stream);
    void* ptrs[] = {x->d_sensors, x->d_doppler_wrap, x->d_export, x->d_export_valid, x->d_move, x->d_tracks, x->d_scenes, x->d_track_ring, x->d_uring, x->d_keypoints, x->d_default_posture,
                    x->d_assoc, x->d_labels, x->d_counters, x->d_phase, x->d_defer, x->d_scene_stats, x->d_ring_hist,
                    x->d_results[0], x->d_results[1], x->d_blob, x->d_bn1s,
                    x->d_bn1t, x->d_bn2s, x->d_bn2t, x->d_feats, x->d_row_scene, x->d_row_track, x->d_row_slot,
                    x->d_pose_total, x->d_act2, x->d_act3, x->d_pose_out, x->d_row_scene2, x->d_row_track2, x->d_row_slot2,
                    x->d_pose_total2, x->d_pose_extra};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    pose_tc_free(&x->tc);
    if (x->h_defer_hint) cudaFreeHost(x->h_defer_hint);
    if (x->h_rows_hint) cudaFreeHost(x->h_rows_hint);
    for (int i = 0; i < 2; ++i) {
        const StageSlot& s = x->stage[i];
        for (void* p : {(void*)s.pts, (void*)s.offsets, (void*)s.dt, (void*)s.pk})
            if (p) cudaFree(p);
        for (cudaEvent_t e : {s.uploaded, s.free, x->packed[i], x->results_done[i], x->feat_done[i], x->packt_done[i],
                              x->pose_done[i]})
            if (e) cudaEventDestroy(e);
    }
    if (x->h2d_stream) cudaStreamDestroy(x->h2d_stream);
    if (x->d2h_stream) cudaStreamDestroy(x->d2h_stream);
    if (x->pose_stream) { cudaStreamSynchronize(x->pose_stream); cudaStreamDestroy(x->pose_stream); }
    if (x->stream) cudaStreamDestroy(x->stream);
    delete x;
    return MMW_OK;
}

int mmw_reset(mmw_ctx* x) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    if (x->pose_stream) CK(join_pose(x));
    x->pipe_r = -1;
    x->last_pose_run = 0;
    CK(cudaMemsetAsync(x->d_scenes, 0, sizeof(SceneRec) * x->S, x->stream));
    CK(cudaMemsetAsync(x->d_tracks, 0, sizeof(TrackRec) * (size_t)x->S * x->tcap, x->stream));
    CK(cudaMemsetAsync(x->d_counters, 0, sizeof(unsigned long long) * 8, x->stream));
    CK(cudaMemsetAsync(x->d_assoc, 0xff, sizeof(int32_t) * (size_t)x->S * x->ncap, x->stream));
    CK(cudaMemsetAsync(x->d_pose_total, 0, sizeof(int), x->stream));
    CK(cudaMemsetAsync(x->d_pose_total2, 0, sizeof(int), x->stream));
    CK(cudaMemsetAsync(x->d_pose_extra, 0, 2 * sizeof(int32_t), x->stream));
    CK(cudaMemsetAsync(x->d_defer, 0, sizeof(int32_t) * (2 + 2 * (size_t)x->S), x->stream));
    CK(cudaMemsetAsync(x->d_scene_stats, 0, sizeof(int32_t) * 8 * (size_t)x->S, x->stream));
    CK(cudaMemsetAsync(x->d_ring_hist, 0, (size_t)kRing * kHistBytes * x->S, x->stream));
    return MMW_OK;
}

// ---- checkpoint / resume -------------------------------------------------------------------------
namespace {
struct StateHeader {
    uint32_t magic, abi;
    int32_t S, ncap, tcap, ring_size;
    uint64_t bytes;
};
constexpr uint32_t kStateMagic = 0x4d4d5753u;   // "MMWS"
struct StatePart { void* dev; size_t bytes; };
// Every part is [S][...]: a scene blob record holds each part's per-scene slice, in this order.
enum { kPartScene, kPartTracks, kPartTrackRing, kPartURing, kPartHist, kPartKeypoints, kPartPoseCnt, kNumStateParts };
std::vector<StatePart> state_parts(mmw_ctx* x) {
    const size_t S = x->S;
    return {{x->d_scenes, sizeof(SceneRec) * S},
            {x->d_tracks, sizeof(TrackRec) * S * x->tcap},
            {x->d_track_ring, sizeof(float) * S * x->tcap * kRing * kFeatPts * kRawCols},
            {x->d_uring, sizeof(float) * S * kRing * x->ncap * kRawCols},
            {x->d_ring_hist, (size_t)kRing * kHistBytes * S},
            {x->d_keypoints, sizeof(float) * S * x->tcap * kKp},
            {x->d_defer + 1 + S, sizeof(int32_t) * S}};                 // pose rows per scene of the last frame
}
}  // namespace

size_t mmw_state_size(mmw_ctx* x) {
    if (!x) return 0;
    size_t n = sizeof(StateHeader);
    for (const StatePart& p : state_parts(x)) n += p.bytes;
    return n;
}

int mmw_state_dump(mmw_ctx* x, void* host_blob, size_t bytes) {
    if (!x || !host_blob) return fail(MMW_ERR_INVALID, "ctx/host_blob is NULL");
    const size_t need = mmw_state_size(x);
    if (bytes < need) return fail(MMW_ERR_CAPACITY, "state blob buffer is smaller than mmw_state_size()");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    StateHeader h{kStateMagic, MMW_ABI_VERSION, x->S, x->ncap, x->tcap, x->dc.ring_size, (uint64_t)need};
    unsigned char* o = static_cast<unsigned char*>(host_blob);
    std::memcpy(o, &h, sizeof(h));
    o += sizeof(h);
    for (const StatePart& p : state_parts(x)) {
        CK(cudaMemcpy(o, p.dev, p.bytes, cudaMemcpyDeviceToHost));
        o += p.bytes;
    }
    return MMW_OK;
}

int mmw_state_restore(mmw_ctx* x, const void* host_blob, size_t bytes) {
    if (!x || !host_blob) return fail(MMW_ERR_INVALID, "ctx/host_blob is NULL");
    StateHeader h;
    if (bytes < sizeof(h)) return fail(MMW_ERR_INVALID, "state blob is truncated");
    std::memcpy(&h, host_blob, sizeof(h));
    if (h.magic != kStateMagic || h.abi != MMW_ABI_VERSION)
        return fail(MMW_ERR_INVALID, "not a state blob of this library version");
    if (h.S != x->S || h.ncap != x->ncap || h.tcap != x->tcap || h.ring_size != x->dc.ring_size)
        return fail(MMW_ERR_INVALID, "state blob was taken from a context of another shape "
                                     "(n_scenes / max_points_per_frame / max_tracks / frames_batch)");
    if (h.bytes != mmw_state_size(x) || bytes < h.bytes) return fail(MMW_ERR_INVALID, "state blob is truncated");
    CK(cudaSetDevice(x->device));
    CK(mmw_sync(x) == MMW_OK ? cudaSuccess : cudaErrorUnknown);
    const unsigned char* o = static_cast<const unsigned char*>(host_blob) + sizeof(h);
    for (const StatePart& p : state_parts(x)) {
        CK(cudaMemcpy(p.dev, o, p.bytes, cudaMemcpyHostToDevice));
        o += p.bytes;
    }
    return MMW_OK;
}

int mmw_create(const mmw_config* cfg, int device, int n_scenes, int max_points, int max_tracks, mmw_ctx** out) {
    if (!cfg || !out) return fail(MMW_ERR_INVALID, "cfg/out is NULL");
    if (n_scenes < 1 || max_points < 1 || max_tracks < 1 || max_tracks > kMaxTcap)
        return fail(MMW_ERR_INVALID, "n_scenes >= 1, max_points >= 1, 1 <= max_tracks <= 32 required");
    if (cfg->frames_batch < 0 || cfg->frames_batch > kRing - 1)
        return fail(MMW_ERR_INVALID, "frames_batch must be 0..2");
    if (cfg->xyz_q_format < 0 || cfg->xyz_q_format > 15) return fail(MMW_ERR_INVALID, "xyz_q_format must be 0..15");
    if (cfg->db_min_samples < 1 || cfg->tr_max_tracks < 0)
        return fail(MMW_ERR_INVALID, "db_min_samples >= 1 and tr_max_tracks >= 0 required");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(MMW_ERR_CUDA, "no such CUDA device");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int smem = step_smem_bytes(max_points, max_tracks);
    if ((size_t)smem > prop.sharedMemPerBlockOptin || (size_t)dbscan_big_smem_bytes(max_points) > prop.sharedMemPerBlockOptin)
        return fail(MMW_ERR_CAPACITY, "max_points/max_tracks need more shared memory than one CTA can have");
    mmw_ctx* x = new (std::nothrow) mmw_ctx();
    if (!x) return fail(MMW_ERR_INVALID, "out of host memory");
    x->cfg = *cfg;
    x->device = device; x->S = n_scenes; x->ncap = max_points; x->tcap = max_tracks;
    fill_devconfig(*cfg, max_points, max_tracks, &x->dc);
    const size_t S = n_scenes;
#define ALLOC(p, bytes)                                                       \
    do {                                                                      \
        cudaError_t e__ = cudaMalloc((void**)&(p), (bytes));                  \
        if (e__ != cudaSuccess) {                                             \
            mmw_destroy(x);                                                   \
            return fail(MMW_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e__)); \
        }                                                                     \
    } while (0)
    if (cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete x;
        return fail(MMW_ERR_CUDA, "cudaStreamCreate failed");
    }
    ALLOC(x->d_tracks, sizeof(TrackRec) * S * max_tracks);
    ALLOC(x->d_scenes, sizeof(SceneRec) * S);
    ALLOC(x->d_track_ring, sizeof(float) * S * max_tracks * kRing * kFeatPts * kRawCols);
    ALLOC(x->d_uring, sizeof(float) * S * kRing * max_points * kRawCols);
    ALLOC(x->d_keypoints, sizeof(float) * S * max_tracks * kKp);
    ALLOC(x->d_default_posture, sizeof(float) * kKp);
    ALLOC(x->d_assoc, sizeof(int32_t) * S * max_points);
    ALLOC(x->d_labels, sizeof(int32_t) * S * 3 * max_points);
    ALLOC(x->d_counters, sizeof(unsigned long long) * 8);
    ALLOC(x->d_phase, sizeof(unsigned long long) * (16 + 3 * S + 16));
    ALLOC(x->d_defer, sizeof(int32_t) * (2 + 2 * S));
    ALLOC(x->d_scene_stats, sizeof(int32_t) * 8 * S);
    if (cudaHostAlloc((void**)&x->h_defer_hint, sizeof(int32_t), cudaHostAllocMapped) == cudaSuccess) {
        *x->h_defer_hint = 0;
        if (cudaHostGetDevicePointer((void**)&x->d_defer_hint, x->h_defer_hint, 0) != cudaSuccess) x->d_defer_hint = nullptr;
    } else {
        (void)cudaGetLastError();
        x->h_defer_hint = nullptr;
    }
    if (cudaHostAlloc((void**)&x->h_rows_hint, sizeof(int32_t), cudaHostAllocMapped) == cudaSuccess) {
        *x->h_rows_hint = 0;
        if (cudaHostGetDevicePointer((void**)&x->d_rows_hint, x->h_rows_hint, 0) != cudaSuccess) x->d_rows_hint = nullptr;
    } else {
        (void)cudaGetLastError();
        x->h_rows_hint = nullptr;
    }
    ALLOC(x->d_ring_hist, (size_t)kRing * kHistBytes * S);
    {
        const char* env = getenv("MMW_POSE_INDEX_FOLD");
        x->fold_pose_index = S <= 4096 && !(env && env[0] == '0');
    }
    for (int i = 0; i < 2; ++i) {
        StageSlot& st = x->stage[i];
        st.pts_cap = sizeof(float) * kRawCols * S * max_points + kStageSlack;      // one full frame (run_frames grows it)
        ALLOC(st.pts, st.pts_cap);
        ALLOC(st.offsets, sizeof(int32_t) * kGroup * (S + 1));
        ALLOC(st.dt, sizeof(double) * kGroup * S);
        ALLOC(x->d_results[i], sizeof(float) * S * max_tracks * MMW_RESULT_FLOATS);
        if (cudaEventCreateWithFlags(&st.uploaded, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&st.free, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x->packed[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x->results_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x->feat_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x->packt_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&x->pose_done[i], cudaEventDisableTiming) != cudaSuccess) {
            mmw_destroy(x);
            return fail(MMW_ERR_CUDA, "cudaEventCreate failed");
        }
    }
    // the pose network is the critical path of the throughput mode: its CTAs are scheduled ahead of the tracker's
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithFlags(&x->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithPriority(&x->pose_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithFlags(&x->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) {
        mmw_destroy(x);
        return fail(MMW_ERR_CUDA, "cudaStreamCreate failed");
    }
    ALLOC(x->d_pose_total, sizeof(int));
    ALLOC(x->d_pose_extra, 2 * sizeof(int32_t));
    x->pose_cap = n_scenes * max_tracks;
    ALLOC(x->d_row_scene, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_row_track, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_row_slot, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_row_scene2, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_row_track2, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_row_slot2, sizeof(int32_t) * x->pose_cap);
    ALLOC(x->d_pose_total2, sizeof(int));
    ALLOC(x->d_feats, sizeof(float) * (size_t)x->pose_cap * kRing * kFeatPts * kRawCols);
    ALLOC(x->d_pose_out, sizeof(float) * (size_t)x->pose_cap * kKp);
    ALLOC(x->d_sensors, sizeof(SensorRec) * S);
    ALLOC(x->d_doppler_wrap, sizeof(double) * S);
#undef ALLOC
    cudaMemcpy(x->d_default_posture, cfg->default_posture, sizeof(float) * kKp, cudaMemcpyHostToDevice);
    x->sensors.assign(S, config_sensor(*cfg));
    {
        const std::vector<SensorRec> recs(S, x->dc.sensor);
        const std::vector<double> wrap(S, doppler_wrap(x->sensors[0]));
        if (cudaMemcpy(x->d_sensors, recs.data(), sizeof(SensorRec) * S, cudaMemcpyHostToDevice) != cudaSuccess ||
            cudaMemcpy(x->d_doppler_wrap, wrap.data(), sizeof(double) * S, cudaMemcpyHostToDevice) != cudaSuccess) {
            mmw_destroy(x);
            return fail(MMW_ERR_CUDA, "upload of the sensor table failed");
        }
    }
    cudaMemset(x->d_keypoints, 0, sizeof(float) * S * max_tracks * kKp);
    int rc = mmw_reset(x);
    if (rc != MMW_OK) { mmw_destroy(x); return rc; }
    sync_main(x);
    *out = x;
    return MMW_OK;
}

// Queues the upload of table entries first .. first + n - 1 on the context's stream, behind all work queued there (the
// previous frame's feature kernel included, which runs on this stream in throughput mode too).  Nothing on the pose
// stream reads the table: dense 2's fade-square epilogue uses only the context-wide window geometry.  The sources are
// pageable vectors, which cudaMemcpyAsync stages before it returns.
static int upload_sensors(mmw_ctx* x, int first, int n) {
    std::vector<SensorRec> recs(n);
    std::vector<double> wrap(n);
    for (int i = 0; i < n; ++i) {
        recs[i] = sensor_rec(x->sensors[first + i]);
        wrap[i] = doppler_wrap(x->sensors[first + i]);
    }
    CK(cudaSetDevice(x->device));
    CK(cudaMemcpyAsync(x->d_sensors + first, recs.data(), sizeof(SensorRec) * n, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(x->d_doppler_wrap + first, wrap.data(), sizeof(double) * n, cudaMemcpyHostToDevice, x->stream));
    return MMW_OK;
}

int mmw_set_doppler_resolution(mmw_ctx* x, double doppler_res) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    if (!(doppler_res > 0.0) || !std::isfinite(doppler_res)) return fail(MMW_ERR_INVALID, "doppler_res must be positive and finite");
    x->cfg.doppler_res = doppler_res;
    x->dc.sensor.doppler_res = doppler_res;
    for (mmw_scene_sensor& p : x->sensors) p.doppler_res = doppler_res;
    return upload_sensors(x, 0, x->S);
}

// What is wrong with a sensor-table entry, or nullptr: the rules of mmw_set_scene_sensors.
static const char* sensor_error(const mmw_scene_sensor& p) {
    if (!std::isfinite(p.s_height) || !std::isfinite(p.s_tilt_deg) || !std::isfinite(p.z_max) ||
        !std::isfinite(p.doppler_res))
        return "sensor parameters must be finite";
    if (!(p.doppler_res > 0.0)) return "doppler_res must be positive";
    if (p.xyz_q_format < 0 || p.xyz_q_format > 15) return "xyz_q_format must be 0..15";
    if (p.num_doppler_bins < 0) return "num_doppler_bins must not be negative";
    return nullptr;
}

int mmw_set_scene_sensors(mmw_ctx* x, int first, int n, const mmw_scene_sensor* params) {
    if (!x || !params) return fail(MMW_ERR_INVALID, "ctx/params is NULL");
    if (first < 0 || n < 0 || n > x->S - first) return fail(MMW_ERR_INVALID, "scene range out of bounds");
    for (int i = 0; i < n; ++i)
        if (const char* e = sensor_error(params[i])) return fail(MMW_ERR_INVALID, e);
    if (n == 0) return MMW_OK;
    for (int i = 0; i < n; ++i) x->sensors[first + i] = params[i];
    return upload_sensors(x, first, n);
}

int mmw_get_scene_sensors(mmw_ctx* x, int first, int n, mmw_scene_sensor* out) {
    if (!x || !out) return fail(MMW_ERR_INVALID, "ctx/out is NULL");
    if (first < 0 || n < 0 || n > x->S - first) return fail(MMW_ERR_INVALID, "scene range out of bounds");
    for (int i = 0; i < n; ++i) out[i] = x->sensors[first + i];
    return MMW_OK;
}

// MMW_OK, or MMW_ERR_INVALID for a list of n scene indices with one out of range or listed twice.
static int check_scene_list(const mmw_ctx* x, const int32_t* scenes, int n) {
    if (n < 0) return fail(MMW_ERR_INVALID, "n must not be negative");
    std::vector<char> seen(x->S, 0);
    for (int i = 0; i < n; ++i) {
        const int s = scenes[i];
        if (s < 0 || s >= x->S) return fail(MMW_ERR_INVALID, "scene index out of range");
        if (seen[s]) return fail(MMW_ERR_INVALID, "scene index listed twice");
        seen[s] = 1;
    }
    return MMW_OK;
}

int mmw_reset_scenes(mmw_ctx* x, const int32_t* scenes, int n) {
    if (!x || (!scenes && n > 0)) return fail(MMW_ERR_INVALID, "ctx/scenes is NULL");
    const int rc = check_scene_list(x, scenes, n);
    if (rc != MMW_OK) return rc;
    CK(cudaSetDevice(x->device));
    if (x->pose_stream) CK(join_pose(x));
    int32_t* pose_cnt = x->d_defer + 1 + x->S;       // StepArgs::pose_cnt
    for (int i = 0; i < n; ++i) {
        const size_t s = scenes[i];
        CK(cudaMemsetAsync(x->d_scenes + s, 0, sizeof(SceneRec), x->stream));
        CK(cudaMemsetAsync(x->d_tracks + s * x->tcap, 0, sizeof(TrackRec) * x->tcap, x->stream));
        CK(cudaMemsetAsync(x->d_ring_hist + s * kRing * kHistBytes, 0, (size_t)kRing * kHistBytes, x->stream));
        CK(cudaMemsetAsync(x->d_scene_stats + s * 8, 0, sizeof(int32_t) * 8, x->stream));
        CK(cudaMemsetAsync(pose_cnt + s, 0, sizeof(int32_t), x->stream));
    }
    return MMW_OK;
}

int mmw_sync(mmw_ctx* x) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(cudaStreamSynchronize(x->h2d_stream));
    CK(sync_main(x));
    CK(cudaStreamSynchronize(x->d2h_stream));
    return MMW_OK;
}

void* mmw_stream(mmw_ctx* x) { return x ? (void*)x->stream : nullptr; }
uint64_t mmw_launch_count(mmw_ctx* x) { return x ? x->launches : 0; }

// ------------------------------------------------------------------------------------------------
int mmw_load_pose_weights(mmw_ctx* x, int variant, const float* blob, size_t n) {
    if (!x || !blob) return fail(MMW_ERR_INVALID, "ctx/blob is NULL");
    if (variant != MMW_POSE_2D && variant != MMW_POSE_3D) return fail(MMW_ERR_INVALID, "unknown pose variant");
    const int D = variant == MMW_POSE_3D ? 3 : 1;
    if (D != x->dc.ring_size)
        return fail(MMW_ERR_INVALID, "pose variant does not match frames_batch (2-D net needs frames_batch=0, "
                                     "3-D net needs frames_batch=2; Utils.py:517-520)");
    const int taps = D == 3 ? 27 : 9;
    const int Kf = D * 64 * 32, H = D * 512;
    const size_t sz[16] = {(size_t)taps * 5 * 16, 16, (size_t)taps * 16 * 32, 32, 32, 32, 32, 32,
                           (size_t)Kf * H, (size_t)H, (size_t)H, (size_t)H, (size_t)H, (size_t)H,
                           (size_t)H * kKp, (size_t)kKp};
    size_t off[17];
    off[0] = 0;
    for (int i = 0; i < 16; ++i) off[i + 1] = off[i] + sz[i];
    if (n != off[16]) return fail(MMW_ERR_INVALID, "weight blob has the wrong number of floats for this variant");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    x->has_weights = false;              // a failed reload must not leave the old pointers in use
    x->last_pose_run = 0;
    if (x->d_blob) { cudaFree(x->d_blob); x->d_blob = nullptr; }
    for (float** p : {&x->d_bn1s, &x->d_bn1t, &x->d_bn2s, &x->d_bn2t, &x->d_act2, &x->d_act3})
        if (*p) { cudaFree(*p); *p = nullptr; }
    CK(cudaMalloc((void**)&x->d_blob, sizeof(float) * n));
    CK(cudaMemcpy(x->d_blob, blob, sizeof(float) * n, cudaMemcpyHostToDevice));
    x->w1 = x->d_blob + off[0]; x->b1 = x->d_blob + off[1];
    x->w2 = x->d_blob + off[2]; x->b2 = x->d_blob + off[3];
    x->wd1 = x->d_blob + off[8]; x->bd1 = x->d_blob + off[9];
    x->wd2 = x->d_blob + off[14]; x->bd2 = x->d_blob + off[15];
    // BatchNorm at inference (Keras, eps = 1e-3): y = gamma (v - mean)/sqrt(var + eps) + beta = v*scale + shift
    auto bn = [&](size_t g, int cnt, float** ds, float** dt) -> int {
        std::vector<float> sc(cnt), sh(cnt);
        for (int i = 0; i < cnt; ++i) {
            const float gamma = blob[off[g] + i], beta = blob[off[g + 1] + i], mean = blob[off[g + 2] + i],
                        var = blob[off[g + 3] + i];
            const float s = gamma / std::sqrt(var + 1e-3f);
            sc[i] = s;
            sh[i] = beta - mean * s;
        }
        if (cudaMalloc((void**)ds, sizeof(float) * cnt) != cudaSuccess) return -1;
        if (cudaMalloc((void**)dt, sizeof(float) * cnt) != cudaSuccess) return -1;
        cudaMemcpy(*ds, sc.data(), sizeof(float) * cnt, cudaMemcpyHostToDevice);
        cudaMemcpy(*dt, sh.data(), sizeof(float) * cnt, cudaMemcpyHostToDevice);
        return 0;
    };
    if (bn(4, 32, &x->d_bn1s, &x->d_bn1t) || bn(10, H, &x->d_bn2s, &x->d_bn2t))
        return fail(MMW_ERR_CUDA, "cudaMalloc failed for BatchNorm constants");
    CK(cudaMalloc((void**)&x->d_act2, sizeof(float) * (size_t)x->pose_cap * Kf));
    CK(cudaMalloc((void**)&x->d_act3, sizeof(float) * (size_t)x->pose_cap * H));
    x->variant = variant; x->D = D; x->Kf = Kf; x->H = H;
    int rc = pose_tc_init(&x->tc, blob, off, D, x->pose_cap);
    if (rc != 0) return fail(MMW_ERR_CUDA, std::string("tensor-core dense path init failed: ") + pose_tc_error());
    x->has_weights = true;
    return MMW_OK;
}

// Tensor-core path: conv1 -> conv2 -> dense1 -> dense2 on stream st, input buffer b, operands handed over as split
// bf16 (pose_tc.cu).  before_fc2: an event dense 2 waits for (throughput mode: the frame's result records are packed).
static int run_pose_tc(mmw_ctx* x, const PoseTcRun& r, int max_rows, int b, cudaStream_t st,
                       cudaEvent_t before_fc2 = nullptr) {
    const bool marks = st == x->stream;       // the per-kernel events are recorded on the context's stream
    int nl = 0;
    if (marks) prof_mark(x, MMW_K_CONV);
    if (pose_tc_conv(&x->tc, r, st, &nl, b) != 0) return fail(MMW_ERR_CUDA, std::string("tensor-core conv: ") + pose_tc_error());
    x->launches += nl;
    if (marks) prof_mark(x, MMW_K_FC1);
    if (pose_tc_fc1(&x->tc, r, max_rows, st, &nl, x->h_rows_hint ? *(volatile int32_t*)x->h_rows_hint : 0) != 0)
        return fail(MMW_ERR_CUDA, std::string("tensor-core dense 1: ") + pose_tc_error());
    x->launches += nl;
    if (before_fc2) CK(cudaStreamWaitEvent(st, before_fc2, 0));
    if (marks) prof_mark(x, MMW_K_FC2);
    if (pose_tc_fc2(&x->tc, r, max_rows, st, &nl) != 0) return fail(MMW_ERR_CUDA, std::string("tensor-core dense 2: ") + pose_tc_error());
    x->launches += nl;
    if (marks) prof_mark(x, -1);
    return MMW_OK;
}

static int run_pose_net(mmw_ctx* x, float* keypoints_by_slot, int max_rows) {
    x->last_pose_run = x->use_tc && x->tc.ready ? 1 : 2;
    if (x->use_tc && x->tc.ready) {
        PoseTcRun r{x->d_pose_total, x->b1, x->b2, x->d_bn1s, x->d_bn1t, x->bd1, x->d_bn2s, x->d_bn2t, x->bd2,
                    x->d_pose_out, keypoints_by_slot, x->d_row_scene, x->d_row_slot, x->tcap};
        return run_pose_tc(x, r, max_rows, 0, x->stream);
    }
    // CUDA-core fp32 path (kept for numerics comparison)
    ConvArgs ca{x->d_feats, x->w1, x->b1, x->w2, x->b2, x->d_bn1s, x->d_bn1t, x->d_act2, x->d_pose_total};
    int grid = max_rows < 296 ? max_rows : 296;
    prof_mark(x, MMW_K_CONV);
    CK(launch_conv(ca, x->D, grid, x->stream));
    x->launches++;
    FcArgs fa{x->d_act2, x->wd1, x->bd1, x->d_bn2s, x->d_bn2t, x->d_act3, x->d_pose_total, x->Kf, x->H};
    prof_mark(x, MMW_K_FC1);
    CK(launch_fc1_simt(fa, max_rows, x->stream));
    x->launches++;
    Fc2Args f2{x->d_act3, x->wd2, x->bd2, x->d_pose_out, keypoints_by_slot, x->d_row_scene, x->d_row_slot,
               x->d_pose_total, x->H, x->tcap};
    grid = (max_rows + 7) / 8 < 148 * 4 ? (max_rows + 7) / 8 : 148 * 4;
    prof_mark(x, MMW_K_FC2);
    CK(launch_fc2(f2, grid, x->stream));
    x->launches++;
    prof_mark(x, -1);
    return MMW_OK;
}

// Throughput mode, the part of a step after the tracker (MMW_STEP_PIPELINE).  Frame k, buffers b = k & 1:
//   main stream : [step k][dbscan_big k] (queued by the caller)  wait pose(k-2)  [features k -> inputs b]  ev feat[b]
//                 wait pose(k-1)  [pack_tracks k -> results b]  ev packt[b]                    ... then frame k+1
//   pose stream : wait feat[b]  [conv1][conv2][dense 1]  wait packt[b]  [dense 2 -> keypoints, results b]  ev pose[b]
// so the tracker of frame k+1 runs under the convolutions / dense 1 of frame k.  The pose stream is serial, hence
// "pose(k-1) done" implies every earlier frame's pose work is done (its activations are single-buffered).
static int pipeline_pose(mmw_ctx* x);
static int estimate_posture_impl(mmw_ctx* x, bool late);
static int launch_pack_tracks(mmw_ctx* x, float* results);

// The feature stage on stream st: the pose-row scan (unless pose_feature_kernel folds it in), then the feature maps,
// the packed tensor-core input of buffer b and the row maps of buffer b.  late: the feature kernel lays out the rows of
// the tracks step_kernel left and does not wait for dbscan_big_kernel, which appends the rows of the tracks it spawns.
static int launch_feature_stage(mmw_ctx* x, int b, bool late, cudaStream_t st) {
    int* pose_total = b ? x->d_pose_total2 : x->d_pose_total;
    if (!x->fold_pose_index) {
        prof_mark(x, MMW_K_POSE_INDEX);
        CK(launch_pose_index(x->d_scenes, x->S, pose_total, x->d_counters, st));
        x->launches++;
    }
    PoseFeatArgs fa{x->dc, x->d_sensors, x->d_scenes, x->d_tracks, x->d_track_ring, x->d_feats,
                    (x->use_tc && x->tc.ready) ? pose_tc_input(&x->tc, b) : nullptr, b ? x->d_row_scene2 : x->d_row_scene,
                    b ? x->d_row_track2 : x->d_row_track, b ? x->d_row_slot2 : x->d_row_slot,
                    x->fold_pose_index ? x->d_defer + 1 + x->S : nullptr, pose_total, x->d_counters, x->S};
    fa.rows_hint = x->d_rows_hint;
    fa.late_extra = late ? x->d_pose_extra + b : nullptr;
    x->rows_buf = b;
    prof_mark(x, MMW_K_POSE_FEATURES);
    CK(launch_pose_features(fa, x->S, st));
    x->launches++;
    return MMW_OK;
}

// The flag checks of every step entry point, made before anything is queued.
static int check_step_flags(const mmw_ctx* x, uint32_t flags) {
    if ((flags & MMW_STEP_POSE) && !x->has_weights)
        return fail(MMW_ERR_STATE, "MMW_STEP_POSE needs mmw_load_pose_weights first");
    if ((flags & MMW_STEP_PIPELINE) && (!(flags & MMW_STEP_POSE) || !(x->use_tc && x->tc.ready)))
        return fail(MMW_ERR_STATE, "MMW_STEP_PIPELINE needs MMW_STEP_POSE and the tensor-core pose path");
    if ((flags & MMW_STEP_PIPELINE) && (flags & MMW_STEP_RECORD_LABELS))
        return fail(MMW_ERR_INVALID, "MMW_STEP_PIPELINE cannot record labels");
    return MMW_OK;
}

// The number of rows of a frame's offsets [S+1], or -1 unless offsets[0] == 0 and they do not decrease.
static long long offsets_total(const int32_t* offsets, int S) {
    if (offsets[0] != 0) return -1;
    for (int i = 0; i < S; ++i)
        if (offsets[i] > offsets[i + 1]) return -1;
    return offsets[S];
}

// ---- input staging: a ring of two slots, filled on the upload stream so that the upload of the next step (or group
// of frames) overlaps the kernels of this one.  A slot is free once the steps that read it have run.  That event is
// recorded at the head of the NEXT acquire, where the main stream has to wait for an upload anyway -- not behind a
// step's last kernel, where it would sit between dense 2 and the result pack and undo their dependent launch.

static cudaError_t grow(void** buf, size_t* cap, size_t bytes) {
    if (bytes <= *cap) return cudaSuccess;
    cudaError_t e = cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    if (e == cudaSuccess && (e = cudaMalloc(buf, bytes)) == cudaSuccess) *cap = bytes;
    return e;
}

// Takes the next slot (*k) for pts_bytes of point rows and pk_bytes of packets, and makes the upload stream wait until
// the slot is free.  A slot that is too small is reallocated once the steps that last read it are done.
static int stage_acquire(mmw_ctx* x, size_t pts_bytes, size_t pk_bytes, int* k) {
    for (int i = 0; i < 2; ++i)
        if (x->stage_pending & (1u << i)) CK(cudaEventRecord(x->stage[i].free, x->stream));
    x->stage_pending = 0;
    *k = (int)(x->stage_idx++ & 1u);
    StageSlot& s = x->stage[*k];
    if (pts_bytes + kStageSlack > s.pts_cap || pk_bytes > s.pk_cap) {
        CK(cudaEventSynchronize(s.free));
        CK(grow((void**)&s.pts, &s.pts_cap, pts_bytes + kStageSlack));
        CK(grow((void**)&s.pk, &s.pk_cap, pk_bytes));
    }
    CK(cudaStreamWaitEvent(x->h2d_stream, s.free, 0));
    return MMW_OK;
}

// The slot's uploads are queued: the main stream waits for them.
static int stage_submit(mmw_ctx* x, int k) {
    CK(cudaEventRecord(x->stage[k].uploaded, x->h2d_stream));
    CK(cudaStreamWaitEvent(x->stream, x->stage[k].uploaded, 0));
    return MMW_OK;
}

// Every step that reads the slot is queued: its free event is recorded by the next stage_acquire.
static void stage_release(mmw_ctx* x, int k) { x->stage_pending |= 1u << k; }

static int step_queue(mmw_ctx* x, StepArgs& a, uint32_t flags);

int mmw_step(mmw_ctx* x, const float* pts, const int32_t* offsets, const double* dt, uint32_t flags) {
    if (!x || !offsets || !dt) return fail(MMW_ERR_INVALID, "ctx/offsets/dt is NULL");
    if ((flags & MMW_STEP_DEVICE_INPUT) && !pts) return fail(MMW_ERR_INVALID, "pts is NULL");
    int rc = check_step_flags(x, flags);
    if (rc != MMW_OK) return rc;
    CK(cudaSetDevice(x->device));
    StepArgs a;
    if (flags & MMW_STEP_DEVICE_INPUT) {
        a.pts = pts; a.offsets = offsets; a.dt = dt;
        return step_queue(x, a, flags);
    }
    const long long total = offsets_total(offsets, x->S);
    if (total < 0) return fail(MMW_ERR_INVALID, "offsets must start at 0 and must not decrease");
    if (total > (long long)x->S * x->ncap)
        return fail(MMW_ERR_CAPACITY, "more points than n_scenes * max_points_per_frame");
    if (total > 0 && !pts) return fail(MMW_ERR_INVALID, "pts is NULL");
    const size_t bytes = ((flags & MMW_STEP_INPUT_I16) ? sizeof(int16_t) : sizeof(float)) * kRawCols * total;
    int k;
    if ((rc = stage_acquire(x, bytes, 0, &k)) != MMW_OK) return rc;
    const StageSlot& s = x->stage[k];
    if (total) CK(cudaMemcpyAsync(s.pts, pts, bytes, cudaMemcpyHostToDevice, x->h2d_stream));
    CK(cudaMemcpyAsync(s.offsets, offsets, sizeof(int32_t) * (x->S + 1), cudaMemcpyHostToDevice, x->h2d_stream));
    CK(cudaMemcpyAsync(s.dt, dt, sizeof(double) * x->S, cudaMemcpyHostToDevice, x->h2d_stream));
    if ((rc = stage_submit(x, k)) != MMW_OK) return rc;
    a.pts = s.pts; a.offsets = s.offsets; a.dt = s.dt;
    rc = step_queue(x, a, flags);
    stage_release(x, k);
    return rc;
}

// The tracker kernels of a step whose inputs a.pts / a.offsets / a.dt / a.pts_row0 are in place, then its pose stage.
// The flags have passed check_step_flags.
static int step_queue(mmw_ctx* x, StepArgs& a, uint32_t flags) {
    a.cfg = x->dc;
    a.sensors = x->d_sensors;
    a.tracks = x->d_tracks; a.scenes = x->d_scenes; a.track_ring = x->d_track_ring; a.uring = x->d_uring;
    a.keypoints = x->d_keypoints; a.default_posture = x->d_default_posture; a.assoc_out = x->d_assoc;
    a.labels_out = (flags & MMW_STEP_RECORD_LABELS) ? x->d_labels : nullptr;
    a.counters = x->d_counters; a.n_scenes = x->S; a.flags = flags;
    a.phase_cycles = x->phase_clocks ? x->d_phase : nullptr;
    a.defer_count = x->d_defer;
    a.defer_done = x->d_defer + 1 + 2 * x->S;
    a.defer_list = x->d_defer + 1;
    a.pose_cnt = x->d_defer + 1 + x->S;
    a.scene_stats = x->d_scene_stats;
    a.defer_hint = x->d_defer_hint;
    a.ring_hist = x->d_ring_hist;
    const bool pipelined = (flags & MMW_STEP_PIPELINE) != 0;
    // fused serial steps on the tensor-core pose path: the feature kernel does not wait for dbscan_big_kernel, which
    // appends the rows of the tracks it spawns itself (StepArgs::nr_*, buffer 0).  In throughput mode, where the pose
    // network of the previous frame holds most SMs, this measured 2 % slower -- 0.2324 against 0.2274 ms per step --
    // and 1.7 % faster in serial mode, 0.2419 against 0.2461.
    const bool late = !pipelined && (flags & MMW_STEP_POSE) && x->fold_pose_index && x->use_tc && x->tc.ready;
    if (late) {
        a.nr_feats = x->d_feats;
        a.nr_packed = pose_tc_input(&x->tc);
        a.nr_row_scene = x->d_row_scene;
        a.nr_row_track = x->d_row_track;
        a.nr_row_slot = x->d_row_slot;
        a.nr_extra = x->d_pose_extra;
    }
    if (pipelined) {
        // frame k-2 used the same pose inputs / row maps (buffer k & 1): its pose network must be done before
        // dbscan_big_kernel appends rows and the feature kernel fills them.  Queued in front of the tracker kernels (not
        // between dbscan_big_kernel and the feature kernel, whose dependent launch it would undo); already satisfied in
        // steady state, the previous frame's pack_tracks waited for the same event.
        if (x->pipe_idx >= 2) CK(cudaStreamWaitEvent(x->stream, x->pose_done[x->pipe_idx & 1u], 0));
    } else {
        CK(join_pose(x));
        x->pipe_r = -1;
    }
    prof_mark(x, MMW_K_STEP);
    CK(launch_step(a, x->stream));
    prof_mark(x, MMW_K_DBSCAN_BIG);
    // one CTA per deferred scene of the last step the device has reported, within [16, 148]
    CK(launch_dbscan_big(a, x->stream, x->h_defer_hint ? *(volatile int32_t*)x->h_defer_hint : 16));
    x->launches += 2;          // step_kernel + dbscan_big_kernel
    prof_mark(x, -1);
    if (pipelined) return pipeline_pose(x);
    if (flags & MMW_STEP_POSE) return estimate_posture_impl(x, late);
    return MMW_OK;
}

int mmw_estimate_posture(mmw_ctx* x) { return estimate_posture_impl(x, false); }

static int estimate_posture_impl(mmw_ctx* x, bool late) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    if (!x->has_weights) return fail(MMW_ERR_STATE, "estimate_posture needs mmw_load_pose_weights first");
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    const int rc = launch_feature_stage(x, 0, late, x->stream);
    if (rc != MMW_OK) return rc;
    return run_pose_net(x, x->d_keypoints, x->pose_cap);
}

int mmw_pose_features_only(mmw_ctx* x) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    x->last_pose_run = 0;                // the network input and the row count now belong to no run
    return launch_feature_stage(x, 0, false, x->stream);
}

int mmw_set_keypoints(mmw_ctx* x, int scene, int track_index, const float* kp57) {
    if (!x || !kp57) return fail(MMW_ERR_INVALID, "NULL argument");
    if (scene < 0 || scene >= x->S || track_index < 0 || track_index >= x->tcap)
        return fail(MMW_ERR_INVALID, "scene/track out of range");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    TrackRec t;
    CK(cudaMemcpy(&t, x->d_tracks + (size_t)scene * x->tcap + track_index, sizeof(t), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(x->d_keypoints + ((size_t)scene * x->tcap + t.slot) * kKp, kp57, sizeof(float) * kKp,
                  cudaMemcpyHostToDevice));
    return MMW_OK;
}

// ------------------------------------------------------------------------------------------------
int mmw_get_tracks(mmw_ctx* x, mmw_track_out* tracks, int32_t* n_tracks) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    std::vector<SceneRec> sc(x->S);
    CK(cudaMemcpy(sc.data(), x->d_scenes, sizeof(SceneRec) * x->S, cudaMemcpyDeviceToHost));
    if (n_tracks)
        for (int s = 0; s < x->S; ++s) n_tracks[s] = sc[s].n_tracks;
    if (!tracks) return MMW_OK;
    std::vector<TrackRec> tr((size_t)x->S * x->tcap);
    std::vector<float> kp((size_t)x->S * x->tcap * kKp);
    CK(cudaMemcpy(tr.data(), x->d_tracks, sizeof(TrackRec) * tr.size(), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(kp.data(), x->d_keypoints, sizeof(float) * kp.size(), cudaMemcpyDeviceToHost));
    for (int s = 0; s < x->S; ++s) {
        for (int k = 0; k < x->tcap; ++k) {
            mmw_track_out& o = tracks[(size_t)s * x->tcap + k];
            std::memset(&o, 0, sizeof(o));
            if (k >= sc[s].n_tracks) { o.id = -1; continue; }
            const TrackRec& t = tr[(size_t)s * x->tcap + k];
            o.id = t.id; o.point_num = t.point_num; o.is_static = t.is_static; o.ring_frames = t.ring_n;
            for (int f = 0; f < kRing; ++f)
                o.ring_counts[f] = f < t.ring_n ? t.ring_cnt[(t.ring_head + f) % x->dc.ring_size] : -1;
            o.lifetime = t.lifetime; o.n_est = t.n_est;
            std::memcpy(o.x, t.x, sizeof(t.x)); std::memcpy(o.P, t.P, sizeof(t.P));
            std::memcpy(o.spread_est, t.spread, sizeof(t.spread));
            std::memcpy(o.group_disp_est, t.G, sizeof(t.G));
            std::memcpy(o.centroid, t.centroid, sizeof(t.centroid));
            std::memcpy(o.min_vals, t.minv, sizeof(t.minv)); std::memcpy(o.max_vals, t.maxv, sizeof(t.maxv));
            std::memcpy(o.keypoints, &kp[((size_t)s * x->tcap + t.slot) * kKp], sizeof(float) * kKp);
        }
    }
    return MMW_OK;
}

int mmw_get_scene_summary(mmw_ctx* x, int32_t* n_tracks, int32_t* next_id, int32_t* last_M) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    std::vector<SceneRec> sc(x->S);
    CK(cudaMemcpyAsync(sc.data(), x->d_scenes, sizeof(SceneRec) * x->S, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    for (int s = 0; s < x->S; ++s) {
        if (n_tracks) n_tracks[s] = sc[s].n_tracks;
        if (next_id) next_id[s] = sc[s].next_id;
        if (last_M) last_M[s] = sc[s].last_M;
    }
    return MMW_OK;
}

int mmw_get_point_assoc(mmw_ctx* x, int32_t* assoc, size_t n) {
    if (!x || !assoc) return fail(MMW_ERR_INVALID, "ctx/assoc is NULL");
    if (n > (size_t)x->S * x->ncap) return fail(MMW_ERR_CAPACITY, "n exceeds n_scenes * max_points_per_frame");
    CK(cudaSetDevice(x->device));
    CK(cudaMemcpyAsync(assoc, x->d_assoc, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    return MMW_OK;
}

int mmw_get_labels(mmw_ctx* x, int32_t* labels, int32_t* n_fused) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    if (labels)
        CK(cudaMemcpy(labels, x->d_labels, sizeof(int32_t) * (size_t)x->S * 3 * x->ncap, cudaMemcpyDeviceToHost));
    if (n_fused) {
        std::vector<SceneRec> sc(x->S);
        CK(cudaMemcpy(sc.data(), x->d_scenes, sizeof(SceneRec) * x->S, cudaMemcpyDeviceToHost));
        for (int s = 0; s < x->S; ++s) n_fused[s] = sc[s].last_ran ? sc[s].dbscan_n : -1;
    }
    return MMW_OK;
}

int mmw_get_status(mmw_ctx* x, uint32_t* flags) {
    if (!x || !flags) return fail(MMW_ERR_INVALID, "ctx/flags is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    std::vector<SceneRec> sc(x->S);
    CK(cudaMemcpy(sc.data(), x->d_scenes, sizeof(SceneRec) * x->S, cudaMemcpyDeviceToHost));
    for (int s = 0; s < x->S; ++s) flags[s] = sc[s].flags;
    return MMW_OK;
}

int mmw_get_ring_counts(mmw_ctx* x, int32_t* counts) {
    if (!x || !counts) return fail(MMW_ERR_INVALID, "ctx/counts is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    std::vector<SceneRec> sc(x->S);
    CK(cudaMemcpy(sc.data(), x->d_scenes, sizeof(SceneRec) * x->S, cudaMemcpyDeviceToHost));
    for (int s = 0; s < x->S; ++s)
        for (int f = 0; f < kRing; ++f)
            counts[s * kRing + f] =
                f < sc[s].ring_n ? sc[s].ring_cnt[(sc[s].ring_head + f) % x->dc.ring_size] : -1;
    return MMW_OK;
}

static int ring_edit(mmw_ctx* x, int scene, bool clear) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    if (scene < 0 || scene >= x->S) return fail(MMW_ERR_INVALID, "scene out of range");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    SceneRec sc;
    CK(cudaMemcpy(&sc, x->d_scenes + scene, sizeof(sc), cudaMemcpyDeviceToHost));
    if (clear) {
        sc.ring_n = 0; sc.ring_head = 0; sc.ring_cnt[0] = sc.ring_cnt[1] = sc.ring_cnt[2] = 0;
        sc.ring_ph_gone = 1;
    } else if (!sc.ring_ph_gone) {       // the deque still starts with its initial empty frame: that is what pops
        sc.ring_ph_gone = 1;
    } else if (sc.ring_n > 0) {          // popleft (Tracking.py:66-71)
        sc.ring_cnt[sc.ring_head] = 0;
        sc.ring_head = (sc.ring_head + 1) % x->dc.ring_size;
        sc.ring_n -= 1;
    }
    CK(cudaMemcpy(x->d_scenes + scene, &sc, sizeof(sc), cudaMemcpyHostToDevice));
    return MMW_OK;
}
int mmw_ring_pop(mmw_ctx* x, int scene) { return ring_edit(x, scene, false); }
int mmw_ring_clear(mmw_ctx* x, int scene) { return ring_edit(x, scene, true); }

int mmw_get_pose_rows(mmw_ctx* x, int32_t* n_rows, int32_t* scene_idx, int32_t* track_idx, float* feats,
                      size_t cap_floats) {
    if (!x || !n_rows) return fail(MMW_ERR_INVALID, "ctx/n_rows is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    const int b = x->rows_buf;
    int n = 0;
    CK(cudaMemcpy(&n, b ? x->d_pose_total2 : x->d_pose_total, sizeof(int), cudaMemcpyDeviceToHost));
    *n_rows = n;
    if (n == 0 || (!scene_idx && !track_idx && !feats)) return MMW_OK;
    // Rows come back in (scene, list index) order.  On the device the rows of tracks spawned this frame lie behind all
    // others (dbscan_big_kernel appends them, in the order its CTAs get there).
    std::vector<int32_t> hs(n), ht(n);
    CK(cudaMemcpy(hs.data(), b ? x->d_row_scene2 : x->d_row_scene, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ht.data(), b ? x->d_row_track2 : x->d_row_track, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int p, int q) { return hs[p] != hs[q] ? hs[p] < hs[q] : ht[p] < ht[q]; });
    for (int i = 0; i < n; ++i) {
        if (scene_idx) scene_idx[i] = hs[order[i]];
        if (track_idx) track_idx[i] = ht[order[i]];
    }
    if (feats) {
        const size_t per = (size_t)x->dc.ring_size * kFeatPts * kRawCols;
        if (cap_floats < per * n) return fail(MMW_ERR_CAPACITY, "feats buffer too small");
        std::vector<float> hf(per * n);
        CK(cudaMemcpy(hf.data(), x->d_feats, sizeof(float) * per * n, cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; ++i) std::memcpy(feats + per * i, hf.data() + per * order[i], sizeof(float) * per);
    }
    return MMW_OK;
}

int mmw_get_counters(mmw_ctx* x, uint64_t out[8], int reset) {
    if (!x || !out) return fail(MMW_ERR_INVALID, "ctx/out is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    unsigned long long h[8];
    CK(cudaMemcpy(h, x->d_counters, sizeof(h), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 8; ++i) out[i] = h[i];
    if (reset) CK(cudaMemset(x->d_counters, 0, sizeof(h)));
    return MMW_OK;
}

}  // extern "C"

// ================================================================================================
// stage-level kernels
// ================================================================================================
namespace mmw {

__global__ void preprocess_kernel(DevConfig c, const float* pts, size_t n, double* world, uint8_t* keep) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = pts + i * kRawCols;
    double w[6];
    world_from_raw(c.sensor, p[0], p[1], p[2], p[3], w);
    double* o = world + i * 8;
#pragma unroll
    for (int k = 0; k < 6; ++k) o[k] = w[k];
    o[6] = __dmul_rn((double)p[3], c.sensor.doppler_res);
    o[7] = (double)p[4];
    keep[i] = ((w[2] <= c.sensor.z_max) && (w[2] > 0.0) && (w[1] > 0.0)) ? 1 : 0;
}

__global__ void __launch_bounds__(kStepThreads) dbscan_stage_kernel(DevConfig c, const double* xyz,
                                                                    const int32_t* offsets, double eps, int min_samples,
                                                                    int32_t* labels, int maxB) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* X = reinterpret_cast<double*>(smem);
    double* Y = X + maxB;
    double* Z = Y + maxB;
    int* par = reinterpret_cast<int*>(Z + maxB);
    int* cl = par + maxB;
    int* scan = cl + maxB;
    const int off = offsets[blockIdx.x];
    const int B = offsets[blockIdx.x + 1] - off;
    if (B <= 0) return;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        X[b] = xyz[(size_t)(off + b) * 3 + 0];
        Y[b] = xyz[(size_t)(off + b) * 3 + 1];
        Z[b] = xyz[(size_t)(off + b) * 3 + 2];
    }
    __syncthreads();
    dbscan_block(NbExact{c, X, Y, Z, eps}, B, min_samples, par, cl, scan);
    for (int b = threadIdx.x; b < B; b += blockDim.x) labels[off + b] = cl[b];
}

// One CTA of 128 threads per track: the element-parallel steps of linalg.cuh, as the fused step kernel runs them.
__global__ void __launch_bounds__(128) kalman_predict_kernel(double* x, double* P, const double* dt, int n, double q_var) {
    __shared__ double sx[9], sP[81];
    const int i = blockIdx.x, tid = threadIdx.x;
    const Elem el(tid);
    if (tid < 81) sP[tid] = P[(size_t)i * 81 + tid];
    if (tid < 9) sx[tid] = x[(size_t)i * 9 + tid];
    __syncthreads();
    const double pv = tid < 81 ? kf_predict_elem(sP, dt[i], q_var, el) : 0.0;
    const double xn = tid < 9 ? kf_predict_x(sx, dt[i], tid) : 0.0;
    if (tid < 81) P[(size_t)i * 81 + tid] = pv;
    if (tid < 9) x[(size_t)i * 9 + tid] = xn;
}

__global__ void __launch_bounds__(128) kalman_update_kernel(double* x, double* P, const double* z, const double* R,
                                                            const uint8_t* life0, int n, double thres, double gain) {
    __shared__ double sx[9], sP[81], sz[6], sR[36], sS[36], sM1[81], sK[54], sKR[54];
    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const Elem el(tid);
    if (tid < 81) sP[tid] = P[(size_t)i * 81 + tid];
    if (tid < 36) sR[tid] = R[(size_t)i * 36 + tid];
    if (tid < 9) sx[tid] = x[(size_t)i * 9 + tid];
    if (tid < 6) sz[tid] = z[(size_t)i * 6 + tid];
    __syncthreads();
    if (tid < 36) sS[tid] = sP[el.i6 * 9 + el.a6] + sR[tid];          // S = P[:6,:6] + R
    __syncthreads();
    if (warp == 0) {
        double r[6];
        (void)inv6_spd_half(lane < 16 ? sS : nullptr, lane, r);
        __syncwarp();
        if (lane >= 6 && lane < 12) {
#pragma unroll
            for (int k = 0; k < 6; ++k) sS[k * 6 + (lane - 6)] = r[k];
        }
    }
    __syncthreads();
    if (tid < 54) sK[tid] = kf_update_K_elem(sP, sS, el);
    __syncthreads();
    if (tid < 81) sM1[tid] = kf_update_M1_elem(sP, sK, el);
    if (tid < 54) sKR[tid] = kf_update_KR_elem(sK, sR, el);
    if (warp == 3) {
        const double xv = lane < 9 ? kf_update_x(sx, sz, sK, lane) : 0.0;
        __syncwarp();
        if (lane < 9) sx[lane] = xv;
    }
    __syncthreads();
    if (tid < 81) sP[tid] = kf_update_P_elem(sM1, sK, sKR, el);
    if (tid == 96) kf_update_nudge(sx, sz, life0[i] != 0, thres, gain);
    __syncthreads();
    if (tid < 81) P[(size_t)i * 81 + tid] = sP[tid];
    if (tid < 9) x[(size_t)i * 9 + tid] = sx[tid];
}

__global__ void __launch_bounds__(128) gate_stage_kernel(const double* pts, int M, const double* hx, const double* C,
                                                         int T, double gate, double* d2, int32_t* assoc) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* gp = reinterpret_cast<double*>(smem);             // [T][kGateWords]
    double* sC = gp + (size_t)T * kGateWords;                 // [T][36]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int e = threadIdx.x; e < T * 36; e += blockDim.x) sC[e] = C[e];
    for (int e = threadIdx.x; e < T * 6; e += blockDim.x) gp[(e / 6) * kGateWords + 21 + e % 6] = hx[e];
    __syncthreads();
    for (int j0 = 0; j0 < T; j0 += 8) {
        const int j = j0 + 2 * warp + (lane >> 4);
        const bool live = j < T;
        if (__ballot_sync(kFull, live) == 0u) continue;
        double r[6];
        const double det = inv6_spd_half(live ? sC + j * 36 : nullptr, lane, r);
        if (live) gate_pack_half(gp + j * kGateWords, r, det, lane);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
        double w[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) w[k] = pts[(size_t)i * 6 + k];
        double best = INFINITY;
        int bj = -1;
        for (int j = 0; j < T; ++j) {
            const double v = gate_score(gp + j * kGateWords, w);
            d2[(size_t)i * T + j] = v;
            if (v < gate && v < best) { best = v; bj = j; }
        }
        assoc[i] = bj;
    }
}

// ---- UART TLV packets -> fp32 point rows (ReadDataIWR1443.py:88-201) ------------------------------------
// The header walk runs on the host too (mmw_step_packets): one definition for both.
constexpr int kTlvHeader = 36;
__host__ __device__ __forceinline__ uint32_t rd_u32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__host__ __device__ __forceinline__ int rd_i16(const uint8_t* p) {
    return (int)(int16_t)((uint16_t)p[0] | ((uint16_t)p[1] << 8));
}

// Number of objects a packet yields (0 when the reference would return dataOK = 0) and its frame number.
__host__ __device__ __forceinline__ int tlv_packet_objects(const uint8_t* p, long long len, int* frame) {
    const uint8_t magic[8] = {2, 1, 4, 3, 6, 5, 8, 7};
    *frame = 0;
    if (len < kTlvHeader) return 0;
    for (int i = 0; i < 8; ++i)
        if (p[i] != magic[i]) return 0;
    const uint32_t total = rd_u32(p + 12);
    if ((unsigned long long)len < total) return 0;                       // incomplete packet (:81-83)
    *frame = (int)rd_u32(p + 20);
    if (rd_u32(p + 28) == 0) return 0;                                   // numDetectedObj (:106)
    if (len < kTlvHeader + 12) return 0;
    if (rd_u32(p + kTlvHeader) != 1u) return 0;                          // MMWDEMO_UART_MSG_DETECTED_POINTS (:115)
    const int n_obj = (int)((uint32_t)p[kTlvHeader + 8] | ((uint32_t)p[kTlvHeader + 9] << 8));
    if (len < kTlvHeader + 12 + 12LL * n_obj) return 0;
    return n_obj;
}

__global__ void tlv_count_kernel(const uint8_t* bytes, const long long* off, int n, int32_t* counts, int32_t* frames) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int fr;
    counts[i] = tlv_packet_objects(bytes + off[i], off[i + 1] - off[i], &fr);
    frames[i] = fr;
}

// One warp per packet, one lane per object (12 bytes in, 20 bytes out).  The dopplerIdx threshold is half_bins_m1, or
// half_bins_m1_s[packet] when that is given (one radar profile per scene).
__global__ void __launch_bounds__(256) tlv_decode_kernel(const uint8_t* bytes, const long long* off, int n,
                                                         const int32_t* point_off, double half_bins_m1,
                                                         const double* half_bins_m1_s, double doppler_res,
                                                         float* points) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const int n_obj = point_off[w + 1] - point_off[w];
    if (n_obj == 0) return;
    if (half_bins_m1_s) half_bins_m1 = half_bins_m1_s[w];
    const uint8_t* p = bytes + off[w];
    const int q = (int)((uint32_t)p[kTlvHeader + 10] | ((uint32_t)p[kTlvHeader + 11] << 8));
    const double scale = exp2((double)q);                                // 2 ** xyzQFormat (:126-128)
    const uint8_t* body = p + kTlvHeader + 12;
    float* o = points + (size_t)point_off[w] * kRawCols;
    for (int j = lane; j < n_obj; j += 32) {
        const uint8_t* b = body + 12 * j;
        int dop = rd_i16(b + 2);
        if ((double)dop > half_bins_m1) dop = (int)(int16_t)(dop - 65535);   // :167-175 on int16 data (numpy 1.26 wrap)
        o[j * kRawCols + 0] = (float)((double)rd_i16(b + 6) / scale);
        o[j * kRawCols + 1] = (float)((double)rd_i16(b + 8) / scale);
        o[j * kRawCols + 2] = (float)((double)rd_i16(b + 10) / scale);
        o[j * kRawCols + 3] = (float)((double)dop * doppler_res);        // doppler_res: in units of the context's (1 = the index)
        o[j * kRawCols + 4] = (float)rd_i16(b + 4);
    }
}

// Dataset-builder export of track 0 (preprocessing.py:185-216; Utils.relative_coordinates :437-465 and
// format_batched_frames :523-548): ring frames newest first, [x - cx, y - cy, z, doppler, peakVal] of the first 64
// rows per frame in float64, zero padded, unsorted, raw intensity.  One CTA of 64 threads per scene.
constexpr int kExportRows = kRing * kFeatPts;               // the reference always writes three frames (Utils.py:526)
__global__ void __launch_bounds__(kFeatPts) export_track0_kernel(DevConfig c, const SensorRec* sensors,
                                                                 const SceneRec* scenes, const TrackRec* tracks,
                                                                 const float* track_ring, double* out, int32_t* valid) {
    const int s = blockIdx.x, i = threadIdx.x;
    const SensorRec& sr = sensors[s];
    const SceneRec sc = scenes[s];
    const TrackRec* t = tracks + (size_t)s * c.tcap;
    double* o = out + (size_t)s * (kExportRows * kRawCols + 2);
    bool ok = sc.last_ran && sc.n_tracks > 0 && t->lifetime == 0.0;
    int total = 0;
    if (ok)
        for (int f = 0; f < t->ring_n; ++f) total += t->ring_cnt[(t->ring_head + f) % c.ring_size];
    ok = ok && total > 0;
    if (i == 0) valid[s] = ok ? 1 : 0;
    if (!ok) return;
    const double cx = t->centroid[0], cy = t->centroid[1];
    if (i == 0) { o[kExportRows * kRawCols] = cx; o[kExportRows * kRawCols + 1] = cy; }
    for (int k = 0; k < kRing; ++k) {
        double v[kRawCols] = {0.0, 0.0, 0.0, 0.0, 0.0};
        if (k < t->ring_n) {
            const int phys = (t->ring_head + t->ring_n - 1 - k) % c.ring_size;          // newest frame first
            if (i < t->ring_cnt[phys]) {
                const float* r = track_ring + ((((size_t)s * c.tcap + t->slot) * kRing + phys) * kFeatPts + i) * kRawCols;
                double yw, zw;
                world_yz(sr, (double)r[1], (double)r[2], yw, zw);
                v[0] = __dsub_rn((double)r[0], cx);
                v[1] = __dsub_rn(yw, cy);
                v[2] = zw;
                v[3] = __dmul_rn((double)r[3], sr.doppler_res);
                v[4] = (double)r[4];
            }
        }
#pragma unroll
        for (int q = 0; q < kRawCols; ++q) o[(k * kFeatPts + i) * kRawCols + q] = v[q];
    }
}

// One CTA per scene, one warp per record (8192 one-record CTAs cost 8 us of launch and tail on the main stream).
__global__ void __launch_bounds__(256) pack_results_kernel(const SceneRec* scenes, const TrackRec* tracks,
                                                           const float* keypoints, int S, int tcap, float* out,
                                                           FadeCfg fade) {
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    pdl_wait();                          // the step's last kernel (dense 2 or the tracker) has completed
    pdl_launch_dependents();
    const int nt = scenes[s].n_tracks;
    for (int k = warp; k < tcap; k += nw) {
        float* o = out + ((size_t)s * tcap + k) * MMW_RESULT_FLOATS;
        if (k >= nt) {
            for (int e = lane; e < MMW_RESULT_FLOATS; e += 32) o[e] = e == 0 ? -1.f : (e == 1 ? (float)nt : 0.f);
            continue;
        }
        const TrackRec* t = tracks + (size_t)s * tcap + k;
        const float* kp = keypoints + ((size_t)s * tcap + t->slot) * kKp;
        for (int e = lane; e < 68; e += 32) {
            float v;
            if (e == 0) v = (float)t->id;
            else if (e == 1) v = (float)nt;
            else if (e < 11) v = (float)t->x[e - 2];
            else v = kp[e - 11];
            o[e] = v;
        }
        if (lane == 0) {
            // calc_fade_square (Visualizer.py:14-29), float64 like the reference
            double cx, cz;
            projection_point(fade, t->x[0] + (double)kp[3], t->x[1] + (double)kp[41], (double)kp[22], cx, cz);
            const double size = fmax(fade.smin, fmin(fade.smax, fade.smax - (t->x[1] + (double)kp[12]) * fade.weight));
            o[68] = (float)cx; o[69] = (float)cz; o[70] = (float)size; o[71] = 0.f;
        }
    }
}

// Throughput mode: the tracker's half of the packed result records of a frame -- id, track count, state x, the
// keypoints the track has NOW (the pose network's dense 2 overwrites them for every track that gets a pose row this
// frame), and x[0], x[1] as two float64 in fields 68..71 for dense 2's fade square.  Records of tracks without a pose
// row this frame (scenes whose frame was skipped) are finished here.
__global__ void __launch_bounds__(256) pack_tracks_kernel(const SceneRec* scenes, const TrackRec* tracks,
                                                          const float* keypoints, int tcap, float* out, FadeCfg fade) {
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int nt = scenes[s].n_tracks;
    const bool ran = scenes[s].last_ran != 0;
    for (int k = warp; k < tcap; k += nw) {
        float* o = out + ((size_t)s * tcap + k) * MMW_RESULT_FLOATS;
        if (k >= nt) {
            for (int e = lane; e < MMW_RESULT_FLOATS; e += 32) o[e] = e == 0 ? -1.f : (e == 1 ? (float)nt : 0.f);
            continue;
        }
        const TrackRec* t = tracks + (size_t)s * tcap + k;
        const float* kp = keypoints + ((size_t)s * tcap + t->slot) * kKp;
        for (int e = lane; e < 68; e += 32) {
            float v;
            if (e == 0) v = (float)t->id;
            else if (e == 1) v = (float)nt;
            else if (e < 11) v = (float)t->x[e - 2];
            else v = kp[e - 11];
            o[e] = v;
        }
        if (lane == 0) {
            if (ran) {
                reinterpret_cast<double*>(o + 68)[0] = t->x[0];
                reinterpret_cast<double*>(o + 68)[1] = t->x[1];
            } else {
                write_fade_square(fade, t->x[0], t->x[1], kp, o);
            }
        }
    }
}

// Live records of a frame, compacted in (scene, list index) order, written straight into mapped host memory
// (mmw_run_frames_compact): CTA s adds up the track counts of the scenes before it (field [1] of a scene's first record),
// its warps copy the scene's live records as 16-byte vectors and stamp the scene index into field [71]; the last scene's
// CTA publishes the frame's record count.
__global__ void __launch_bounds__(128) compact_results_kernel(const float* __restrict__ rec, int S, int tcap,
                                                              float* __restrict__ host_out, int32_t* __restrict__ host_count) {
    const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ int wpart[4];
    const size_t scene_stride = (size_t)tcap * MMW_RESULT_FLOATS;
    int part = 0;
    for (int i = threadIdx.x; i < s; i += 128) part += (int)__ldg(rec + (size_t)i * scene_stride + 1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) wpart[warp] = part;
    __syncthreads();
    const int base = wpart[0] + wpart[1] + wpart[2] + wpart[3];
    const int nt = (int)rec[(size_t)s * scene_stride + 1];
    if (s == S - 1 && threadIdx.x == 0) *host_count = base + nt;
    for (int k = warp; k < nt; k += 4) {
        const float4* src = reinterpret_cast<const float4*>(rec + (size_t)s * scene_stride + (size_t)k * MMW_RESULT_FLOATS);
        float4* dst = reinterpret_cast<float4*>(host_out + (size_t)(base + k) * MMW_RESULT_FLOATS);
        if (lane < MMW_RESULT_FLOATS / 4) {
            float4 v = src[lane];
            if (lane == MMW_RESULT_FLOATS / 4 - 1) v.w = (float)s;
            dst[lane] = v;
        }
    }
}

// ---- per-scene export / import (mmw_export_scenes, mmw_import_scenes) ----------------------------------------
// One part of a scene's state: scene s at dev + s * dev_stride, list entry i of the move buffer at buf + i * buf_stride.
// buf == nullptr (scatter only): the scene's bytes are zeroed.  Every size is a multiple of 4 bytes.
struct MovePart {
    unsigned char* dev;
    unsigned char* buf;
    unsigned long long dev_stride, buf_stride;
    unsigned bytes, pad;
};
constexpr int kMaxMoveParts = 10;
struct MoveParts { MovePart p[kMaxMoveParts]; int n; };

// One CTA per listed scene copies all its parts, between the context's state and the move buffer (a device buffer the
// context owns: no kernel touches host memory).  16-byte vectors where both sides and the size allow -- the unassigned
// ring's stride 60 * ncap and the keypoints' 228 * tcap are not always 16-aligned -- 4-byte words otherwise.
template <bool kGather>
__global__ void __launch_bounds__(256) scene_move_kernel(const __grid_constant__ MoveParts m, const int32_t* scenes,
                                                         int S) {
    const int i = blockIdx.x;
    const int s = scenes[i];
    if (s < 0 || s >= S) return;         // the host has validated the list: a second guard only
    for (int k = 0; k < m.n; ++k) {
        const MovePart& p = m.p[k];
        unsigned char* d = p.dev + (size_t)s * p.dev_stride;
        unsigned char* b = p.buf != nullptr ? p.buf + (size_t)i * p.buf_stride : nullptr;
        unsigned char* dst = kGather ? b : d;
        const unsigned char* src = kGather ? d : b;
        if ((((uintptr_t)dst | (uintptr_t)src | p.bytes) & 15) == 0) {
            uint4* o = reinterpret_cast<uint4*>(dst);
            const uint4* q = reinterpret_cast<const uint4*>(src);
            for (unsigned e = threadIdx.x; e < p.bytes / 16; e += blockDim.x) o[e] = q != nullptr ? q[e] : make_uint4(0, 0, 0, 0);
        } else {
            uint32_t* o = reinterpret_cast<uint32_t*>(dst);
            const uint32_t* q = reinterpret_cast<const uint32_t*>(src);
            for (unsigned e = threadIdx.x; e < p.bytes / 4; e += blockDim.x) o[e] = q != nullptr ? q[e] : 0u;
        }
    }
}

}  // namespace mmw

extern "C" {

static FadeCfg fade_cfg(const mmw_ctx* x) {
    return FadeCfg{x->cfg.m_x, x->cfg.m_y, x->cfg.m_z, x->cfg.fade_size_max, x->cfg.fade_size_min, x->cfg.fade_weight};
}

static int launch_pack_tracks(mmw_ctx* x, float* results) {
    pack_tracks_kernel<<<x->S, 256, 0, x->stream>>>(x->d_scenes, x->d_tracks, x->d_keypoints, x->tcap, results, fade_cfg(x));
    CK(cudaGetLastError());
    x->launches++;
    return MMW_OK;
}

static int pipeline_pose(mmw_ctx* x) {
    const int b = (int)(x->pipe_idx & 1u);
    cudaStream_t T = x->stream, P = x->pose_stream;
    x->last_pose_run = 3;
    int rc = launch_feature_stage(x, b, false, T);
    if (rc != MMW_OK) return rc;
    CK(cudaEventRecord(x->feat_done[b], T));
    // the result records of this frame: buffer b must have been downloaded (frame k-2), and the keypoints the tracker
    // side copies are final once frame k-1's pose network is done
    if (cudaEventQuery(x->results_done[b]) != cudaSuccess) {
        (void)cudaGetLastError();
        CK(cudaStreamWaitEvent(T, x->results_done[b], 0));
    }
    if (x->pipe_idx >= 1 && x->pose_pending) CK(cudaStreamWaitEvent(T, x->pose_done[b ^ 1], 0));
    rc = launch_pack_tracks(x, x->d_results[b]);
    if (rc != MMW_OK) return rc;
    CK(cudaEventRecord(x->packt_done[b], T));
    // pose stream
    CK(cudaStreamWaitEvent(P, x->feat_done[b], 0));
    PoseTcRun r{b ? x->d_pose_total2 : x->d_pose_total, x->b1, x->b2, x->d_bn1s, x->d_bn1t, x->bd1, x->d_bn2s, x->d_bn2t,
                x->bd2, x->d_pose_out, x->d_keypoints, b ? x->d_row_scene2 : x->d_row_scene, b ? x->d_row_slot2 : x->d_row_slot,
                x->tcap, x->d_results[b], b ? x->d_row_track2 : x->d_row_track, fade_cfg(x)};
    rc = run_pose_tc(x, r, x->pose_cap, b, P, x->packt_done[b]);
    if (rc != MMW_OK) return rc;
    CK(cudaEventRecord(x->pose_done[b], P));
    x->pose_pending = true;
    x->pipe_r = b;
    x->pipe_idx++;
    return MMW_OK;
}

int mmw_decode_tlv(mmw_ctx* x, const uint8_t* packets, const int64_t* packet_offsets, int n, double num_doppler_bins,
                   double doppler_res, float* points, size_t max_points_total, int32_t* point_offsets,
                   int32_t* frame_numbers, int32_t* data_ok) {
    if (!x || !packet_offsets || !point_offsets || !frame_numbers || !data_ok)
        return fail(MMW_ERR_INVALID, "NULL argument");
    if (n < 0 || packet_offsets[0] != 0) return fail(MMW_ERR_INVALID, "n_packets >= 0 and packet_offsets[0] == 0 required");
    point_offsets[0] = 0;
    if (n == 0) return MMW_OK;
    const size_t nbytes = (size_t)packet_offsets[n];
    if (nbytes && !packets) return fail(MMW_ERR_INVALID, "packets is NULL");
    CK(cudaSetDevice(x->device));
    uint8_t* d_bytes = nullptr; long long* d_off = nullptr; int32_t *d_cnt = nullptr, *d_fr = nullptr, *d_poff = nullptr;
    float* d_pts = nullptr;
    auto cleanup = [&]() { for (void* p : {(void*)d_bytes, (void*)d_off, (void*)d_cnt, (void*)d_fr, (void*)d_poff, (void*)d_pts}) if (p) cudaFree(p); };
#define TLV_CK(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { cleanup(); return fail(MMW_ERR_CUDA, std::string(#expr ": ") + cudaGetErrorString(e__)); } } while (0)
    TLV_CK(cudaMalloc((void**)&d_bytes, nbytes ? nbytes : 1));
    TLV_CK(cudaMalloc((void**)&d_off, sizeof(long long) * (n + 1)));
    TLV_CK(cudaMalloc((void**)&d_cnt, sizeof(int32_t) * n));
    TLV_CK(cudaMalloc((void**)&d_fr, sizeof(int32_t) * n));
    TLV_CK(cudaMalloc((void**)&d_poff, sizeof(int32_t) * (n + 1)));
    TLV_CK(cudaMemcpyAsync(d_bytes, packets, nbytes, cudaMemcpyHostToDevice, x->stream));
    TLV_CK(cudaMemcpyAsync(d_off, packet_offsets, sizeof(long long) * (n + 1), cudaMemcpyHostToDevice, x->stream));
    tlv_count_kernel<<<(n + 255) / 256, 256, 0, x->stream>>>(d_bytes, d_off, n, d_cnt, d_fr);
    TLV_CK(cudaGetLastError());
    std::vector<int32_t> cnt(n);
    TLV_CK(cudaMemcpyAsync(cnt.data(), d_cnt, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, x->stream));
    TLV_CK(cudaMemcpyAsync(frame_numbers, d_fr, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, x->stream));
    TLV_CK(sync_main(x));
    x->launches++;
    size_t total = 0;
    for (int i = 0; i < n; ++i) {
        data_ok[i] = cnt[i] > 0 ? 1 : 0;
        total += (size_t)cnt[i];
        if (total > (size_t)INT32_MAX) { cleanup(); return fail(MMW_ERR_CAPACITY, "more than 2^31 points"); }
        point_offsets[i + 1] = (int32_t)total;
    }
    if (total > max_points_total) { cleanup(); return fail(MMW_ERR_CAPACITY, "points buffer too small for the decoded packets"); }
    if (total > 0) {
        if (!points) { cleanup(); return fail(MMW_ERR_INVALID, "points is NULL"); }
        TLV_CK(cudaMalloc((void**)&d_pts, sizeof(float) * kRawCols * total));
        TLV_CK(cudaMemcpyAsync(d_poff, point_offsets, sizeof(int32_t) * (n + 1), cudaMemcpyHostToDevice, x->stream));
        const long long threads = 32LL * n;
        tlv_decode_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, x->stream>>>(
            d_bytes, d_off, n, d_poff, num_doppler_bins / 2 - 1, nullptr, doppler_res / x->dc.sensor.doppler_res, d_pts);
        TLV_CK(cudaGetLastError());
        x->launches++;
        TLV_CK(cudaMemcpyAsync(points, d_pts, sizeof(float) * kRawCols * total, cudaMemcpyDeviceToHost, x->stream));
        TLV_CK(sync_main(x));
    }
#undef TLV_CK
    cleanup();
    return MMW_OK;
}

int mmw_step_packets(mmw_ctx* x, const uint8_t* packets, const int64_t* packet_offsets, const double* dt, uint32_t flags,
                     int32_t* frame_numbers, int32_t* data_ok) {
    if (!x || !packet_offsets || !dt) return fail(MMW_ERR_INVALID, "ctx/packet_offsets/dt is NULL");
    if (flags & (MMW_STEP_DEVICE_INPUT | MMW_STEP_INPUT_I16))
        return fail(MMW_ERR_INVALID, "mmw_step_packets takes host packets: MMW_STEP_DEVICE_INPUT / MMW_STEP_INPUT_I16 do not apply");
    int rc = check_step_flags(x, flags);
    if (rc != MMW_OK) return rc;
    const int S = x->S;
    if (packet_offsets[0] != 0) return fail(MMW_ERR_INVALID, "packet_offsets[0] must be 0");
    for (int s = 0; s < S; ++s)
        if (packet_offsets[s + 1] < packet_offsets[s]) return fail(MMW_ERR_INVALID, "packet_offsets must be non-decreasing");
    const size_t nbytes = (size_t)packet_offsets[S];
    if (nbytes && !packets) return fail(MMW_ERR_INVALID, "packets is NULL");
    // Headers on the host: dataOK, the frame number and the row layout of every packet (the step needs validated
    // offsets and the capacity check before launch; counting on the device would need a synchronisation).
    std::vector<int32_t> rows(S + 1), frames(S);
    rows[0] = 0;
    const size_t cap = (size_t)S * x->ncap;
    size_t total = 0;
    for (int s = 0; s < S; ++s) {
        int fr = 0;
        const int n_obj = tlv_packet_objects(packets + packet_offsets[s], packet_offsets[s + 1] - packet_offsets[s], &fr);
        if (n_obj > 0 && x->sensors[s].num_doppler_bins == 0)
            return fail(MMW_ERR_STATE, "scene " + std::to_string(s) + ": a packet with objects, but the scene's "
                                       "num_doppler_bins is not set (mmw_set_scene_sensors)");
        total += (size_t)n_obj;
        if (total > cap) return fail(MMW_ERR_CAPACITY, "more points than n_scenes * max_points_per_frame");
        rows[s + 1] = (int32_t)total;
        frames[s] = fr;
    }
    for (int s = 0; s < S; ++s) {
        if (frame_numbers) frame_numbers[s] = frames[s];
        if (data_ok) data_ok[s] = rows[s + 1] > rows[s] ? 1 : 0;
    }
    CK(cudaSetDevice(x->device));
    // [S+1] packet offsets and the packet bytes go into the slot's packet staging, sized for full frames of one
    // detected-points TLV per scene at first use; the row offsets and dt as for mmw_step.
    const size_t off_bytes = sizeof(int64_t) * (S + 1);
    const size_t full = off_bytes + (size_t)S * (kTlvHeader + 12 + 12 * (size_t)x->ncap);
    int k;
    if ((rc = stage_acquire(x, sizeof(float) * kRawCols * total, std::max(off_bytes + nbytes, full), &k)) != MMW_OK) return rc;
    const StageSlot& st = x->stage[k];
    CK(cudaMemcpyAsync(st.pk, packet_offsets, off_bytes, cudaMemcpyHostToDevice, x->h2d_stream));
    if (nbytes) CK(cudaMemcpyAsync(st.pk + off_bytes, packets, nbytes, cudaMemcpyHostToDevice, x->h2d_stream));
    // pageable source: staged before the call returns
    CK(cudaMemcpyAsync(st.offsets, rows.data(), sizeof(int32_t) * (S + 1), cudaMemcpyHostToDevice, x->h2d_stream));
    CK(cudaMemcpyAsync(st.dt, dt, sizeof(double) * S, cudaMemcpyHostToDevice, x->h2d_stream));
    if ((rc = stage_submit(x, k)) != MMW_OK) return rc;
    // Decode straight into the fp32 rows the step reads: rows carry dopplerIdx (factor 1), corrected with each scene's
    // own threshold.
    if (total) {
        prof_mark(x, MMW_K_PACKETS);
        tlv_decode_kernel<<<(unsigned)((32LL * S + 255) / 256), 256, 0, x->stream>>>(
            st.pk + off_bytes, reinterpret_cast<const long long*>(st.pk), S, st.offsets, 0.0, x->d_doppler_wrap, 1.0,
            st.pts);
        CK(cudaGetLastError());
        x->launches++;
        prof_mark(x, -1);
    }
    StepArgs a;
    a.pts = st.pts; a.offsets = st.offsets; a.dt = st.dt;
    rc = step_queue(x, a, flags);
    stage_release(x, k);
    return rc;
}

int mmw_export_track0(mmw_ctx* x, double* rows, int32_t* valid, double* centroid) {
    if (!x || !rows || !valid) return fail(MMW_ERR_INVALID, "ctx/rows/valid is NULL");
    CK(cudaSetDevice(x->device));
    const size_t per = (size_t)kExportRows * kRawCols + 2;
    if (!x->d_export) {
        CK(cudaMalloc((void**)&x->d_export, sizeof(double) * per * x->S));
        CK(cudaMalloc((void**)&x->d_export_valid, sizeof(int32_t) * x->S));
    }
    export_track0_kernel<<<x->S, kFeatPts, 0, x->stream>>>(x->dc, x->d_sensors, x->d_scenes, x->d_tracks, x->d_track_ring,
                                                         x->d_export, x->d_export_valid);
    CK(cudaGetLastError());
    x->launches++;
    std::vector<double> h(per * x->S);
    CK(cudaMemcpyAsync(valid, x->d_export_valid, sizeof(int32_t) * x->S, cudaMemcpyDeviceToHost, x->stream));
    CK(cudaMemcpyAsync(h.data(), x->d_export, sizeof(double) * per * x->S, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    for (int s = 0; s < x->S; ++s) {                               // blocks of invalid scenes are undefined on the device
        double* r = rows + (size_t)s * kExportRows * kRawCols;
        if (valid[s]) std::memcpy(r, h.data() + per * s, sizeof(double) * kExportRows * kRawCols);
        else std::memset(r, 0, sizeof(double) * kExportRows * kRawCols);
        if (centroid) {
            centroid[2 * s] = valid[s] ? h[per * s + kExportRows * kRawCols] : 0.0;
            centroid[2 * s + 1] = valid[s] ? h[per * s + kExportRows * kRawCols + 1] : 0.0;
        }
    }
    return MMW_OK;
}

int mmw_pack_results(mmw_ctx* x, float* device_out) {
    if (!x || !device_out) return fail(MMW_ERR_INVALID, "ctx/device_out is NULL");
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    const FadeCfg fc{x->cfg.m_x, x->cfg.m_y, x->cfg.m_z, x->cfg.fade_size_max, x->cfg.fade_size_min, x->cfg.fade_weight};
    CK(launch_pdl(pack_results_kernel, dim3(x->S), dim3(256), 0, x->stream, dim3(1, 1, 1),
                  (const SceneRec*)x->d_scenes, (const TrackRec*)x->d_tracks, (const float*)x->d_keypoints, x->S, x->tcap,
                  device_out, fc));
    x->launches++;
    return MMW_OK;
}

// ---- per-scene export / import ----------------------------------------------------------------------------------
static size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

// A scene record: the scene's sensor-table entry at 0, then its slice of every state part (kPart* order), each at a
// 16-byte boundary.
struct SceneLayout {
    size_t per[kNumStateParts];          // bytes of the part per scene
    size_t off[kNumStateParts];          // offset of the part in the record
    size_t rec;                          // record bytes, a multiple of 16
};
static SceneLayout scene_layout(mmw_ctx* x) {
    SceneLayout L;
    const std::vector<StatePart> parts = state_parts(x);
    size_t o = align16(sizeof(mmw_scene_sensor));
    for (int k = 0; k < kNumStateParts; ++k) {
        L.per[k] = parts[k].bytes / x->S;
        L.off[k] = o;
        o += align16(L.per[k]);
    }
    L.rec = o;
    return L;
}
static size_t scene_head_bytes(int n) { return sizeof(mmw_scene_blob_header) + align16(sizeof(int32_t) * n); }

// The state parts of the listed scenes <-> the records of the scene blob in the move buffer.
static MoveParts scene_move_parts(mmw_ctx* x, const SceneLayout& L, int n) {
    MoveParts m{};
    const std::vector<StatePart> parts = state_parts(x);
    unsigned char* rec0 = x->d_move + scene_head_bytes(n);
    for (int k = 0; k < kNumStateParts; ++k)
        m.p[m.n++] = MovePart{static_cast<unsigned char*>(parts[k].dev), rec0 + L.off[k], L.per[k], L.rec, (unsigned)L.per[k], 0};
    return m;
}

// The move buffer holds at least `bytes`.  Only called inside the synchronous export / import, after the pose stream
// has joined the main stream: the previous call has finished with the buffer.
static int grow_move(mmw_ctx* x, size_t bytes) {
    CK(grow((void**)&x->d_move, &x->move_cap, bytes));
    return MMW_OK;
}

// What is wrong with a record of a scene blob, or nullptr.  Checked: every field a kernel takes as an index or a count.
//   sensor entry     the rules of mmw_set_scene_sensors (doppler_res > 0, Q format 0..15, ...)
//   SceneRec         0 <= n_tracks <= tcap                    (step_kernel's bulk copy of T0 records, the list)
//                    0 <= ring_n <= ring_size, 0 <= ring_head < ring_size   (ring_wrap, uring / histogram frames)
//                    0 <= ring_cnt[f] <= ncap                 (fused cloud of DBSCAN: at most 3 * ncap rows, labels)
//                    slot_mask = the set of the listed tracks' slots: spawning takes the lowest free slot of
//                      ~slot_mask for each new track, and a spare bit would leave fewer than tcap - n_tracks
//   TrackRec k < n_tracks   0 <= slot < tcap, no two alike  (track ring / keypoints by slot, 1 << slot)
//                    0 <= ring_n <= ring_size, 0 <= ring_head < ring_size, 0 <= ring_cnt[f] <= 64   (feature maps)
//   pose_cnt         0 <= pose_cnt <= tcap                    (prefix sum of pose rows: at most S * tcap rows)
// Not indices or counts: next_id, flags, last_M, last_ran (selects n_tracks), dbscan_n (host only), ring_ph_gone,
// pose_base (rewritten before every read, pose_kernels.cu), the float64 track state, the histogram bytes (summed into
// 16-bit cell counts that only steer the DBSCAN screen) and the rows of the rings.
static const char* scene_record_error(const mmw_ctx* x, const SceneLayout& L, const unsigned char* r) {
    mmw_scene_sensor p;
    std::memcpy(&p, r, sizeof(p));
    if (const char* e = sensor_error(p)) return e;
    const int rs = x->dc.ring_size, tcap = x->tcap, ncap = x->ncap;
    SceneRec sc;
    std::memcpy(&sc, r + L.off[kPartScene], sizeof(sc));
    if (sc.n_tracks < 0 || sc.n_tracks > tcap) return "n_tracks out of range";
    if (sc.ring_n < 0 || sc.ring_n > rs || sc.ring_head < 0 || sc.ring_head >= rs) return "unassigned ring position out of range";
    for (int f = 0; f < kRing; ++f)
        if (sc.ring_cnt[f] < 0 || sc.ring_cnt[f] > ncap) return "unassigned ring count out of range";
    uint32_t used = 0;
    for (int k = 0; k < sc.n_tracks; ++k) {
        TrackRec t;
        std::memcpy(&t, r + L.off[kPartTracks] + sizeof(TrackRec) * k, sizeof(t));
        if (t.slot < 0 || t.slot >= tcap) return "track slot out of range";
        if (used & (1u << t.slot)) return "two tracks hold the same slot";
        used |= 1u << t.slot;
        if (t.ring_n < 0 || t.ring_n > rs || t.ring_head < 0 || t.ring_head >= rs) return "track ring position out of range";
        for (int f = 0; f < kRing; ++f)
            if (t.ring_cnt[f] < 0 || t.ring_cnt[f] > kFeatPts) return "track ring count out of range";
    }
    if (sc.slot_mask != used) return "slot_mask is not the set of the tracks' slots";
    int32_t pose_cnt;
    std::memcpy(&pose_cnt, r + L.off[kPartPoseCnt], sizeof(pose_cnt));
    if (pose_cnt < 0 || pose_cnt > tcap) return "pose-row count out of range";
    return nullptr;
}

size_t mmw_scene_state_size(mmw_ctx* x, int n) {
    if (!x || n < 0) return 0;
    return scene_head_bytes(n) + (size_t)n * scene_layout(x).rec;
}

int mmw_export_scenes(mmw_ctx* x, const int32_t* scenes, int n, void* host_blob, size_t bytes) {
    if (!x || !host_blob || (!scenes && n > 0)) return fail(MMW_ERR_INVALID, "ctx/scenes/host_blob is NULL");
    int rc = check_scene_list(x, scenes, n);
    if (rc != MMW_OK) return rc;
    const size_t need = mmw_scene_state_size(x, n);
    if (bytes < need) return fail(MMW_ERR_CAPACITY, "scene blob buffer is smaller than mmw_scene_state_size()");
    const SceneLayout L = scene_layout(x);
    const size_t head = scene_head_bytes(n);
    std::vector<unsigned char> h(head, 0);
    mmw_scene_blob_header hd{};
    hd.magic = MMW_SCENE_BLOB_MAGIC;
    hd.abi_version = MMW_ABI_VERSION;
    hd.n = n;
    hd.max_points_per_frame = x->ncap;
    hd.max_tracks = x->tcap;
    hd.frames_batch = x->cfg.frames_batch;
    hd.record_bytes = L.rec;
    hd.total_bytes = need;
    std::memcpy(h.data(), &hd, sizeof(hd));
    if (n > 0) std::memcpy(h.data() + sizeof(hd), scenes, sizeof(int32_t) * n);
    unsigned char* o = static_cast<unsigned char*>(host_blob);
    if (n == 0) {
        std::memcpy(o, h.data(), head);
        return MMW_OK;
    }
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    if ((rc = grow_move(x, need)) != MMW_OK) return rc;
    // header and source indices go up with the list the kernel reads; the zero fill makes the padding of the records 0
    CK(cudaMemcpyAsync(x->d_move, h.data(), head, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemsetAsync(x->d_move + head, 0, need - head, x->stream));
    scene_move_kernel<true><<<n, 256, 0, x->stream>>>(scene_move_parts(x, L, n),
                                                     reinterpret_cast<const int32_t*>(x->d_move + sizeof(hd)), x->S);
    CK(cudaGetLastError());
    x->launches++;
    CK(cudaMemcpyAsync(o, x->d_move, need, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    for (int i = 0; i < n; ++i)                          // the sensor table is host state
        std::memcpy(o + head + L.rec * i, &x->sensors[scenes[i]], sizeof(mmw_scene_sensor));
    return MMW_OK;
}

int mmw_import_scenes(mmw_ctx* x, const int32_t* scenes, int n, const void* host_blob, size_t bytes) {
    if (!x || !host_blob || (!scenes && n > 0)) return fail(MMW_ERR_INVALID, "ctx/scenes/host_blob is NULL");
    if (n < 0) return fail(MMW_ERR_INVALID, "n must not be negative");
    mmw_scene_blob_header hd;
    if (bytes < sizeof(hd)) return fail(MMW_ERR_INVALID, "scene blob is truncated");
    std::memcpy(&hd, host_blob, sizeof(hd));
    if (hd.magic != MMW_SCENE_BLOB_MAGIC || hd.abi_version != MMW_ABI_VERSION)
        return fail(MMW_ERR_INVALID, "not a scene blob of this library version");
    if (hd.max_points_per_frame != x->ncap || hd.max_tracks != x->tcap || hd.frames_batch != x->cfg.frames_batch)
        return fail(MMW_ERR_INVALID, "scene blob was exported from a context of another shape "
                                     "(max_points_per_frame / max_tracks / frames_batch)");
    if (hd.n != n) return fail(MMW_ERR_INVALID, "n differs from the scene blob's");
    const SceneLayout L = scene_layout(x);
    const size_t need = mmw_scene_state_size(x, n);
    if (hd.record_bytes != L.rec || hd.total_bytes != need || bytes < need)
        return fail(MMW_ERR_INVALID, "scene blob is truncated or its sizes are inconsistent");
    int rc = check_scene_list(x, scenes, n);
    if (rc != MMW_OK) return rc;
    const size_t head = scene_head_bytes(n);
    const unsigned char* rec0 = static_cast<const unsigned char*>(host_blob) + head;
    std::vector<mmw_scene_sensor> sensors(n);
    for (int i = 0; i < n; ++i) {
        if (const char* e = scene_record_error(x, L, rec0 + L.rec * i))
            return fail(MMW_ERR_INVALID, "scene blob record " + std::to_string(i) + ": " + e);
        std::memcpy(&sensors[i], rec0 + L.rec * i, sizeof(mmw_scene_sensor));
    }
    if (n == 0) return MMW_OK;
    // behind the blob: the destination list, then each scene's SensorRec and Doppler threshold, built on the host
    const size_t idx_bytes = align16(sizeof(int32_t) * n);
    std::vector<SensorRec> recs(n);
    std::vector<double> wrap(n);
    for (int i = 0; i < n; ++i) {
        recs[i] = sensor_rec(sensors[i]);
        wrap[i] = doppler_wrap(sensors[i]);
    }
    std::vector<unsigned char> aux(idx_bytes + (sizeof(SensorRec) + sizeof(double)) * n, 0);
    std::memcpy(aux.data(), scenes, sizeof(int32_t) * n);
    std::memcpy(aux.data() + idx_bytes, recs.data(), sizeof(SensorRec) * n);
    std::memcpy(aux.data() + idx_bytes + sizeof(SensorRec) * n, wrap.data(), sizeof(double) * n);
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    if ((rc = grow_move(x, need + aux.size())) != MMW_OK) return rc;
    unsigned char* a = x->d_move + need;
    CK(cudaMemcpyAsync(x->d_move, host_blob, need, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(a, aux.data(), aux.size(), cudaMemcpyHostToDevice, x->stream));
    MoveParts m = scene_move_parts(x, L, n);
    m.p[m.n++] = MovePart{reinterpret_cast<unsigned char*>(x->d_sensors), a + idx_bytes, sizeof(SensorRec),
                          sizeof(SensorRec), (unsigned)sizeof(SensorRec), 0};
    m.p[m.n++] = MovePart{reinterpret_cast<unsigned char*>(x->d_doppler_wrap), a + idx_bytes + sizeof(SensorRec) * n,
                          sizeof(double), sizeof(double), (unsigned)sizeof(double), 0};
    // the per-scene counters of the last step are cleared, as mmw_reset_scenes clears them
    m.p[m.n++] = MovePart{reinterpret_cast<unsigned char*>(x->d_scene_stats), nullptr, sizeof(int32_t) * 8, 0,
                          (unsigned)(sizeof(int32_t) * 8), 0};
    scene_move_kernel<false><<<n, 256, 0, x->stream>>>(m, reinterpret_cast<const int32_t*>(a), x->S);
    CK(cudaGetLastError());
    x->launches++;
    for (int i = 0; i < n; ++i) x->sensors[scenes[i]] = sensors[i];
    CK(sync_main(x));
    return MMW_OK;
}

// ---- NCCL, bound at run time ---------------------------------------------------------------------------------
namespace {
struct NcclId128 { char b[128]; };          // ncclUniqueId (passed by value to ncclCommInitRank)
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId128, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*CommUserRank)(void*, int*) = nullptr;
    int (*CommCount)(void*, int*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int /* ncclDataType_t */, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);      // the copy this process already uses
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW);
        if (h) {
            api.lib = h;
            *(void**)&api.GetUniqueId = dlsym(h, "ncclGetUniqueId");
            *(void**)&api.CommInitRank = dlsym(h, "ncclCommInitRank");
            *(void**)&api.CommDestroy = dlsym(h, "ncclCommDestroy");
            *(void**)&api.CommUserRank = dlsym(h, "ncclCommUserRank");
            *(void**)&api.CommCount = dlsym(h, "ncclCommCount");
            *(void**)&api.AllGather = dlsym(h, "ncclAllGather");
            *(void**)&api.GetErrorString = dlsym(h, "ncclGetErrorString");
            if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.CommUserRank || !api.CommCount ||
                !api.AllGather)
                api.lib = nullptr;
        }
    }
    return api.lib ? &api : nullptr;
}
int nccl_fail(NcclApi* a, const char* what, int rc) {
    return fail(MMW_ERR_CUDA, std::string(what) + ": " + (a->GetErrorString ? a->GetErrorString(rc) : "NCCL error"));
}
}  // namespace

int mmw_nccl_unique_id(void* id128) {
    if (!id128) return fail(MMW_ERR_INVALID, "id128 is NULL");
    NcclApi* a = nccl_api();
    if (!a) return fail(MMW_ERR_STATE, "libnccl.so.2 is not available in this process");
    const int rc = a->GetUniqueId(id128);
    return rc == 0 ? MMW_OK : nccl_fail(a, "ncclGetUniqueId", rc);
}

int mmw_nccl_comm_init(mmw_ctx* x, const void* id128, int nranks, int rank, void** comm_out) {
    if (!x || !id128 || !comm_out) return fail(MMW_ERR_INVALID, "NULL argument");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(MMW_ERR_INVALID, "bad nranks/rank");
    NcclApi* a = nccl_api();
    if (!a) return fail(MMW_ERR_STATE, "libnccl.so.2 is not available in this process");
    CK(cudaSetDevice(x->device));
    NcclId128 id;
    std::memcpy(id.b, id128, sizeof(id.b));
    void* comm = nullptr;
    const int rc = a->CommInitRank(&comm, nranks, id, rank);
    if (rc != 0) return nccl_fail(a, "ncclCommInitRank", rc);
    *comm_out = comm;
    return MMW_OK;
}

int mmw_nccl_comm_destroy(void* comm) {
    if (!comm) return MMW_OK;
    NcclApi* a = nccl_api();
    if (!a) return fail(MMW_ERR_STATE, "libnccl.so.2 is not available in this process");
    const int rc = a->CommDestroy(comm);
    return rc == 0 ? MMW_OK : nccl_fail(a, "ncclCommDestroy", rc);
}

int mmw_gather_nccl(mmw_ctx* x, void* comm, int nranks, float* device_out_all) {
    if (!x || !comm || !device_out_all) return fail(MMW_ERR_INVALID, "NULL argument");
    NcclApi* a = nccl_api();
    if (!a) return fail(MMW_ERR_STATE, "libnccl.so.2 is not available in this process");
    int rank = -1, count = 0, rc;
    if ((rc = a->CommUserRank(comm, &rank)) != 0) return nccl_fail(a, "ncclCommUserRank", rc);
    if ((rc = a->CommCount(comm, &count)) != 0) return nccl_fail(a, "ncclCommCount", rc);
    if (count != nranks) return fail(MMW_ERR_INVALID, "nranks does not match the communicator");
    const size_t per_rank = (size_t)x->S * x->tcap * MMW_RESULT_FLOATS;
    int prc = mmw_pack_results(x, device_out_all + per_rank * rank);      // straight into this rank's block
    if (prc != MMW_OK) return prc;
    rc = a->AllGather(device_out_all + per_rank * rank, device_out_all, per_rank, /* ncclFloat32 */ 7, comm, x->stream);
    if (rc != 0) return nccl_fail(a, "ncclAllGather", rc);
    return MMW_OK;
}

// The download of a frame's records on the d2h stream: all of them by a copy, or (dev_out != nullptr: the device
// alias of mapped host memory) only the live ones by compact_results_kernel.
static int queue_download(mmw_ctx* x, int r, float* host_out, float* dev_out, int32_t* dev_count) {
    if (dev_out != nullptr) {
        compact_results_kernel<<<x->S, 128, 0, x->d2h_stream>>>(x->d_results[r], x->S, x->tcap, dev_out, dev_count);
        CK(cudaGetLastError());
        x->launches++;
    } else {
        CK(cudaMemcpyAsync(host_out, x->d_results[r], sizeof(float) * (size_t)x->S * x->tcap * MMW_RESULT_FLOATS,
                           cudaMemcpyDeviceToHost, x->d2h_stream));
    }
    return MMW_OK;
}

static int read_results_impl(mmw_ctx* x, float* host_out, int* slot, float* dev_out, int32_t* dev_count);

int mmw_read_results_async(mmw_ctx* x, float* host_out, int* slot) {
    if (!x || !host_out) return fail(MMW_ERR_INVALID, "ctx/host_out is NULL");
    return read_results_impl(x, host_out, slot, nullptr, nullptr);
}

static int read_results_impl(mmw_ctx* x, float* host_out, int* slot, float* dev_out, int32_t* dev_count) {
    CK(cudaSetDevice(x->device));
    if (x->pipe_r >= 0) {
        // throughput mode: the last step produced its own records in d_results[pipe_r]; they are complete when that
        // frame's dense 2 is
        const int r = x->pipe_r;
        CK(cudaStreamWaitEvent(x->d2h_stream, x->pose_done[r], 0));
        const int rc = queue_download(x, r, host_out, dev_out, dev_count);
        if (rc != MMW_OK) return rc;
        CK(cudaEventRecord(x->results_done[r], x->d2h_stream));
        if (slot) *slot = r;
        return MMW_OK;
    }
    CK(join_pose(x));
    const int r = (int)(x->result_idx++ & 1u);
    // The previous download of this buffer must have finished.  In a pipelined loop the host has already waited for
    // it (mmw_wait_results two frames ago), and then no wait is put into the stream: an event between dense 2 and the
    // pack kernel would undo their programmatic dependent launch.
    if (cudaEventQuery(x->results_done[r]) != cudaSuccess) {
        (void)cudaGetLastError();
        CK(cudaStreamWaitEvent(x->stream, x->results_done[r], 0));
    }
    const FadeCfg fc{x->cfg.m_x, x->cfg.m_y, x->cfg.m_z, x->cfg.fade_size_max, x->cfg.fade_size_min, x->cfg.fade_weight};
    CK(launch_pdl(pack_results_kernel, dim3(x->S), dim3(256), 0, x->stream, dim3(1, 1, 1),
                  (const SceneRec*)x->d_scenes, (const TrackRec*)x->d_tracks, (const float*)x->d_keypoints, x->S, x->tcap,
                  x->d_results[r], fc));
    x->launches++;
    CK(cudaEventRecord(x->packed[r], x->stream));
    CK(cudaStreamWaitEvent(x->d2h_stream, x->packed[r], 0));
    const int rc = queue_download(x, r, host_out, dev_out, dev_count);
    if (rc != MMW_OK) return rc;
    CK(cudaEventRecord(x->results_done[r], x->d2h_stream));
    if (slot) *slot = r;
    return MMW_OK;
}

static int run_frames_impl(mmw_ctx* x, int n_frames, const void* pts, const int64_t* frame_row_offsets, const int32_t* offsets,
                           const double* dt, float* results, int32_t* n_records, bool compact, uint32_t flags);

int mmw_run_frames(mmw_ctx* x, int n_frames, const void* pts, const int64_t* frame_row_offsets, const int32_t* offsets,
                   const double* dt, float* results, uint32_t flags) {
    return run_frames_impl(x, n_frames, pts, frame_row_offsets, offsets, dt, results, nullptr, false, flags);
}

int mmw_run_frames_compact(mmw_ctx* x, int n_frames, const void* pts, const int64_t* frame_row_offsets,
                           const int32_t* offsets, const double* dt, float* results, int32_t* n_records, uint32_t flags) {
    if (!n_records) return fail(MMW_ERR_INVALID, "n_records is NULL");
    return run_frames_impl(x, n_frames, pts, frame_row_offsets, offsets, dt, results, n_records, true, flags);
}

static int run_frames_impl(mmw_ctx* x, int n_frames, const void* pts, const int64_t* frame_row_offsets, const int32_t* offsets,
                           const double* dt, float* results, int32_t* n_records, bool compact, uint32_t flags) {
    if (!x || !frame_row_offsets || !offsets || !dt || !results) return fail(MMW_ERR_INVALID, "NULL argument");
    if (n_frames < 0) return fail(MMW_ERR_INVALID, "n_frames must not be negative");
    if (flags & (MMW_STEP_DEVICE_INPUT | MMW_STEP_RECORD_LABELS))
        return fail(MMW_ERR_INVALID, "mmw_run_frames takes host buffers and does not record labels");
    int rc = check_step_flags(x, flags);
    if (rc != MMW_OK) return rc;
    const size_t row_bytes = (flags & MMW_STEP_INPUT_I16) ? sizeof(int16_t) * kRawCols : sizeof(float) * kRawCols;
    const size_t per_frame = (size_t)x->S * x->tcap * MMW_RESULT_FLOATS;
    // Every frame has its own host buffers, so the host never has to wait for a frame's results before queueing the
    // next one -- the device-side buffers (input staging, pose inputs, result records) are handed over by stream
    // events.  The host only keeps the queue bounded: at most kAhead frames in flight.  (Waiting for frame f-1 before
    // queueing f+1 would put the upload of f+1 behind the download of f-1 and leave the pose stream idle for a
    // third of every frame.  2 to 8 frames in flight measured the same: profiles/r02_e2e_variants2.txt.)
    constexpr int kAhead = 4;
    cudaEvent_t done[kAhead] = {nullptr, nullptr, nullptr, nullptr};
    CK(cudaSetDevice(x->device));
    float* dev_results = nullptr;
    int32_t* dev_counts = nullptr;
    if (compact && n_frames > 0) {
        // the kernel writes the host buffers itself: they must be pinned and mapped into the device's address space
        if (cudaHostGetDevicePointer((void**)&dev_results, results, 0) != cudaSuccess ||
            cudaHostGetDevicePointer((void**)&dev_counts, n_records, 0) != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(MMW_ERR_INVALID, "mmw_run_frames_compact needs results and n_records in pinned (device-mapped) host memory");
        }
    }
    for (int f = 0; f < n_frames; ++f)
        if (frame_row_offsets[f + 1] < frame_row_offsets[f]) return fail(MMW_ERR_INVALID, "frame_row_offsets must not decrease");
    for (int i = 0; i < kAhead; ++i) CK(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
    // The inputs of each group of kGroup frames go up into one staging slot, under the kernels of the group before.
    // The first call grows the slots to kGroup full frames (no re-allocation -- and no device synchronisation -- when a
    // later call brings more points).
    const int n_groups = (n_frames + kGroup - 1) / kGroup;
    const size_t full = (size_t)kGroup * x->S * x->ncap * kRawCols * sizeof(float);
    auto upload_group = [&](int g, int* k) -> int {
        const int f0 = g * kGroup, f1 = std::min(f0 + kGroup, n_frames);
        const size_t bytes = (size_t)(frame_row_offsets[f1] - frame_row_offsets[f0]) * row_bytes;
        if (bytes && !pts) return fail(MMW_ERR_INVALID, "pts is NULL");
        const int rc = stage_acquire(x, std::max(bytes, full), 0, k);
        if (rc != MMW_OK) return rc;
        const StageSlot& s = x->stage[*k];
        if (bytes)
            CK(cudaMemcpyAsync(s.pts, static_cast<const unsigned char*>(pts) + (size_t)frame_row_offsets[f0] * row_bytes,
                               bytes, cudaMemcpyHostToDevice, x->h2d_stream));
        CK(cudaMemcpyAsync(s.offsets, offsets + (size_t)f0 * (x->S + 1), sizeof(int32_t) * (size_t)(f1 - f0) * (x->S + 1),
                           cudaMemcpyHostToDevice, x->h2d_stream));
        CK(cudaMemcpyAsync(s.dt, dt + (size_t)f0 * x->S, sizeof(double) * (size_t)(f1 - f0) * x->S,
                           cudaMemcpyHostToDevice, x->h2d_stream));
        return MMW_OK;
    };
    int k = -1, next = -1;                  // slots of this group and of the next
    rc = n_groups > 0 ? upload_group(0, &next) : MMW_OK;
    for (int f = 0; f < n_frames && rc == MMW_OK; ++f) {
        const int g = f / kGroup, f0 = g * kGroup;
        if (f == f0) {
            if (k >= 0) stage_release(x, k);                // the previous group's last frame is queued
            k = next;
            if ((rc = stage_submit(x, k)) != MMW_OK) break;
            if (g + 1 < n_groups && (rc = upload_group(g + 1, &next)) != MMW_OK) break;
        }
        if (f >= kAhead && cudaEventSynchronize(done[f % kAhead]) != cudaSuccess) { rc = fail(MMW_ERR_CUDA, "cudaEventSynchronize failed"); break; }
        const long long total = offsets_total(offsets + (size_t)f * (x->S + 1), x->S);
        if (total < 0 || total > (long long)x->S * x->ncap || total > frame_row_offsets[f + 1] - frame_row_offsets[f]) {
            rc = fail(MMW_ERR_INVALID, "mmw_run_frames: bad offsets (each frame: 0 = offsets[0] <= ... <= offsets[S] <= its rows, <= S * max_points)");
            break;
        }
        StepArgs a;
        a.pts = x->stage[k].pts;
        a.offsets = x->stage[k].offsets + (size_t)(f - f0) * (x->S + 1);
        a.dt = x->stage[k].dt + (size_t)(f - f0) * x->S;
        a.pts_row0 = frame_row_offsets[f] - frame_row_offsets[f0];
        if ((rc = step_queue(x, a, flags)) != MMW_OK) break;
        rc = read_results_impl(x, results + (size_t)f * per_frame, nullptr, compact ? dev_results + (size_t)f * per_frame : nullptr,
                               compact ? dev_counts + f : nullptr);
        if (rc != MMW_OK) break;
        if (cudaEventRecord(done[f % kAhead], x->d2h_stream) != cudaSuccess) rc = fail(MMW_ERR_CUDA, "cudaEventRecord failed");
    }
    if (k >= 0) stage_release(x, k);
    if (cudaStreamSynchronize(x->d2h_stream) != cudaSuccess && rc == MMW_OK) rc = fail(MMW_ERR_CUDA, "cudaStreamSynchronize failed");
    for (int i = 0; i < kAhead; ++i) cudaEventDestroy(done[i]);
    return rc;
}

int mmw_wait_results(mmw_ctx* x, int slot) {
    if (!x || slot < 0 || slot > 1) return fail(MMW_ERR_INVALID, "bad ctx/slot");
    CK(cudaSetDevice(x->device));
    CK(cudaEventSynchronize(x->results_done[slot]));
    return MMW_OK;
}

int mmw_preprocess(mmw_ctx* x, const float* pts, size_t n, double* world, uint8_t* keep) {
    if (!x || !world || !keep || (n && !pts)) return fail(MMW_ERR_INVALID, "NULL argument");
    if (n == 0) return MMW_OK;
    CK(cudaSetDevice(x->device));
    float* dp; double* dw; uint8_t* dk;
    CK(cudaMalloc((void**)&dp, n * kRawCols * sizeof(float)));
    CK(cudaMalloc((void**)&dw, n * 8 * sizeof(double)));
    CK(cudaMalloc((void**)&dk, n));
    CK(cudaMemcpyAsync(dp, pts, n * kRawCols * sizeof(float), cudaMemcpyHostToDevice, x->stream));
    preprocess_kernel<<<(unsigned)((n + 255) / 256), 256, 0, x->stream>>>(x->dc, dp, n, dw, dk);
    CK(cudaGetLastError());
    x->launches++;
    CK(cudaMemcpyAsync(world, dw, n * 8 * sizeof(double), cudaMemcpyDeviceToHost, x->stream));
    CK(cudaMemcpyAsync(keep, dk, n, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    cudaFree(dp); cudaFree(dw); cudaFree(dk);
    return MMW_OK;
}

int mmw_dbscan(mmw_ctx* x, const double* xyz, const int32_t* offsets, int n_clouds, double eps, int min_samples,
               int32_t* labels) {
    if (!x || !offsets || !labels || n_clouds < 0) return fail(MMW_ERR_INVALID, "NULL argument");
    if (n_clouds == 0) return MMW_OK;
    const size_t total = (size_t)offsets[n_clouds];
    int maxB = 0;
    for (int i = 0; i < n_clouds; ++i) {
        const int b = offsets[i + 1] - offsets[i];
        if (b < 0) return fail(MMW_ERR_INVALID, "offsets must be non-decreasing");
        if (b > maxB) maxB = b;
    }
    if (maxB > 3 * x->ncap) return fail(MMW_ERR_CAPACITY, "a cloud has more than 3*max_points points");
    if (total == 0) return MMW_OK;
    if (!xyz) return fail(MMW_ERR_INVALID, "xyz is NULL");
    if (eps <= 0) eps = x->cfg.db_eps;
    if (min_samples <= 0) min_samples = x->cfg.db_min_samples;
    CK(cudaSetDevice(x->device));
    double* dx; int32_t *doff, *dl;
    CK(cudaMalloc((void**)&dx, total * 3 * sizeof(double)));
    CK(cudaMalloc((void**)&doff, (n_clouds + 1) * sizeof(int32_t)));
    CK(cudaMalloc((void**)&dl, total * sizeof(int32_t)));
    CK(cudaMemcpyAsync(dx, xyz, total * 3 * sizeof(double), cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(doff, offsets, (n_clouds + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, x->stream));
    const size_t smem = (size_t)maxB * (3 * 8 + 2 * 4) + 64;
    CK(cudaFuncSetAttribute(dbscan_stage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dbscan_stage_kernel<<<n_clouds, kStepThreads, smem, x->stream>>>(x->dc, dx, doff, eps, min_samples, dl, maxB);
    CK(cudaGetLastError());
    x->launches++;
    CK(cudaMemcpyAsync(labels, dl, total * sizeof(int32_t), cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    cudaFree(dx); cudaFree(doff); cudaFree(dl);
    return MMW_OK;
}

int mmw_kalman_predict(mmw_ctx* x, double* hx, double* hP, const double* dt, int n) {
    if (!x || !hx || !hP || !dt || n < 0) return fail(MMW_ERR_INVALID, "NULL argument");
    if (n == 0) return MMW_OK;
    CK(cudaSetDevice(x->device));
    double *dx, *dP, *ddt;
    CK(cudaMalloc((void**)&dx, (size_t)n * 9 * 8));
    CK(cudaMalloc((void**)&dP, (size_t)n * 81 * 8));
    CK(cudaMalloc((void**)&ddt, (size_t)n * 8));
    CK(cudaMemcpyAsync(dx, hx, (size_t)n * 9 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(dP, hP, (size_t)n * 81 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(ddt, dt, (size_t)n * 8, cudaMemcpyHostToDevice, x->stream));
    kalman_predict_kernel<<<n, 128, 0, x->stream>>>(dx, dP, ddt, n, x->dc.q_var);
    CK(cudaGetLastError());
    x->launches++;
    CK(cudaMemcpyAsync(hx, dx, (size_t)n * 9 * 8, cudaMemcpyDeviceToHost, x->stream));
    CK(cudaMemcpyAsync(hP, dP, (size_t)n * 81 * 8, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    cudaFree(dx); cudaFree(dP); cudaFree(ddt);
    return MMW_OK;
}

int mmw_kalman_update(mmw_ctx* x, double* hx, double* hP, const double* z, const double* R, const uint8_t* life0,
                      int n) {
    if (!x || !hx || !hP || !z || !R || !life0 || n < 0) return fail(MMW_ERR_INVALID, "NULL argument");
    if (n == 0) return MMW_OK;
    CK(cudaSetDevice(x->device));
    double *dx, *dP, *dz, *dR; uint8_t* dl;
    CK(cudaMalloc((void**)&dx, (size_t)n * 9 * 8));
    CK(cudaMalloc((void**)&dP, (size_t)n * 81 * 8));
    CK(cudaMalloc((void**)&dz, (size_t)n * 6 * 8));
    CK(cudaMalloc((void**)&dR, (size_t)n * 36 * 8));
    CK(cudaMalloc((void**)&dl, (size_t)n));
    CK(cudaMemcpyAsync(dx, hx, (size_t)n * 9 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(dP, hP, (size_t)n * 81 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(dz, z, (size_t)n * 6 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(dR, R, (size_t)n * 36 * 8, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(dl, life0, (size_t)n, cudaMemcpyHostToDevice, x->stream));
    kalman_update_kernel<<<n, 128, 0, x->stream>>>(dx, dP, dz, dR, dl, n, x->dc.nudge_thres,
                                                             x->dc.nudge_gain);
    CK(cudaGetLastError());
    x->launches++;
    CK(cudaMemcpyAsync(hx, dx, (size_t)n * 9 * 8, cudaMemcpyDeviceToHost, x->stream));
    CK(cudaMemcpyAsync(hP, dP, (size_t)n * 81 * 8, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    cudaFree(dx); cudaFree(dP); cudaFree(dz); cudaFree(dR); cudaFree(dl);
    return MMW_OK;
}

int mmw_gate(mmw_ctx* x, const double* points, int M, const double* hxv, const double* C, int T, double* d2,
             int32_t* assoc) {
    if (!x || !assoc || M < 0 || T < 0) return fail(MMW_ERR_INVALID, "NULL argument");
    if (M == 0) return MMW_OK;
    if (T > 0 && (!hxv || !C || !d2)) return fail(MMW_ERR_INVALID, "NULL argument");
    if (!points) return fail(MMW_ERR_INVALID, "points is NULL");
    CK(cudaSetDevice(x->device));
    double *dp, *dh = nullptr, *dC = nullptr, *dd = nullptr; int32_t* da;
    CK(cudaMalloc((void**)&dp, (size_t)M * 6 * 8));
    CK(cudaMalloc((void**)&da, (size_t)M * 4));
    CK(cudaMalloc((void**)&dh, (size_t)(T ? T : 1) * 6 * 8));
    CK(cudaMalloc((void**)&dC, (size_t)(T ? T : 1) * 36 * 8));
    CK(cudaMalloc((void**)&dd, (size_t)M * (T ? T : 1) * 8));
    CK(cudaMemcpyAsync(dp, points, (size_t)M * 6 * 8, cudaMemcpyHostToDevice, x->stream));
    if (T) {
        CK(cudaMemcpyAsync(dh, hxv, (size_t)T * 6 * 8, cudaMemcpyHostToDevice, x->stream));
        CK(cudaMemcpyAsync(dC, C, (size_t)T * 36 * 8, cudaMemcpyHostToDevice, x->stream));
    }
    const size_t smem = ((size_t)(T ? T : 1) * (kGateWords + 36)) * 8;
    CK(cudaFuncSetAttribute(gate_stage_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gate_stage_kernel<<<1, 128, smem, x->stream>>>(dp, M, dh, dC, T, x->dc.gate, dd, da);
    CK(cudaGetLastError());
    x->launches++;
    if (T) CK(cudaMemcpyAsync(d2, dd, (size_t)M * T * 8, cudaMemcpyDeviceToHost, x->stream));
    CK(cudaMemcpyAsync(assoc, da, (size_t)M * 4, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    cudaFree(dp); cudaFree(da); cudaFree(dh); cudaFree(dC); cudaFree(dd);
    return MMW_OK;
}

int mmw_pose(mmw_ctx* x, const float* feats, int n, float* keypoints) {
    if (!x || !feats || !keypoints || n < 0) return fail(MMW_ERR_INVALID, "NULL argument");
    if (!x->has_weights) return fail(MMW_ERR_STATE, "mmw_pose needs mmw_load_pose_weights first");
    if (n > x->pose_cap) return fail(MMW_ERR_CAPACITY, "n exceeds n_scenes * max_tracks");
    if (n == 0) return MMW_OK;
    CK(cudaSetDevice(x->device));
    CK(join_pose(x));
    const size_t per = (size_t)x->dc.ring_size * kFeatPts * kRawCols;
    CK(cudaMemcpyAsync(x->d_feats, feats, sizeof(float) * per * n, cudaMemcpyHostToDevice, x->stream));
    CK(cudaMemcpyAsync(x->d_pose_total, &n, sizeof(int), cudaMemcpyHostToDevice, x->stream));
    CK(sync_main(x));     // &n is a stack variable
    if (x->use_tc && x->tc.ready) {
        if (pose_tc_pack_input(&x->tc, x->d_feats, x->d_pose_total, x->stream) != 0)
            return fail(MMW_ERR_CUDA, std::string("tensor-core input pack: ") + pose_tc_error());
        x->launches++;
    }
    int rc = run_pose_net(x, nullptr, n);
    if (rc != MMW_OK) return rc;
    CK(cudaMemcpyAsync(keypoints, x->d_pose_out, sizeof(float) * kKp * n, cudaMemcpyDeviceToHost, x->stream));
    CK(sync_main(x));
    return MMW_OK;
}

int mmw_profile(mmw_ctx* x, int enable) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    for (auto& m : x->marks) cudaEventDestroy(m.first);
    x->marks.clear();
    for (int i = 0; i < MMW_N_KERNELS; ++i) { x->kernel_ms[i] = 0; x->kernel_calls[i] = 0; }
    x->profiling = enable != 0;
    return MMW_OK;
}

int mmw_get_kernel_ms(mmw_ctx* x, double* total_ms, uint64_t* calls) {
    if (!x || !total_ms || !calls) return fail(MMW_ERR_INVALID, "NULL argument");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    for (size_t i = 0; i + 1 < x->marks.size(); ++i) {
        const int k = x->marks[i].second;
        if (k < 0 || k >= MMW_N_KERNELS) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, x->marks[i].first, x->marks[i + 1].first) == cudaSuccess) {
            x->kernel_ms[k] += ms;
            x->kernel_calls[k] += 1;
        }
    }
    for (auto& m : x->marks) cudaEventDestroy(m.first);
    x->marks.clear();
    for (int i = 0; i < MMW_N_KERNELS; ++i) { total_ms[i] = x->kernel_ms[i]; calls[i] = x->kernel_calls[i]; }
    return MMW_OK;
}

int mmw_scene_cycles(mmw_ctx* x, uint64_t* out /*[S]*/) {
    if (!x || !out) return fail(MMW_ERR_INVALID, "NULL argument");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    CK(cudaMemcpy(out, x->d_phase + 16, sizeof(unsigned long long) * 3 * x->S, cudaMemcpyDeviceToHost));
    return MMW_OK;
}

int mmw_dbscan_big_clocks(mmw_ctx* x, uint64_t* out8 /*[16]*/) {
    if (!x || !out8) return fail(MMW_ERR_INVALID, "NULL argument");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    unsigned long long h[16];
    CK(cudaMemcpy(h, x->d_phase + 16 + 3 * x->S, sizeof(h), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 16; ++i) out8[i] = h[i];
    CK(cudaMemset(x->d_phase + 16 + 3 * x->S, 0, sizeof(h)));
    return MMW_OK;
}

int mmw_phase_clocks(mmw_ctx* x, int enable, uint64_t* out16) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    if (out16) {
        unsigned long long h[16];
        CK(cudaMemcpy(h, x->d_phase, sizeof(h), cudaMemcpyDeviceToHost));
        for (int i = 0; i < 16; ++i) out16[i] = h[i];
    }
    CK(cudaMemset(x->d_phase, 0, sizeof(unsigned long long) * 16));
    x->phase_clocks = enable != 0;
    return MMW_OK;
}

/* Test/bench hook: 0 = CUDA-core fp32 dense path, 1 = tcgen05 tensor-core dense path (default). */
int mmw_set_dense_path(mmw_ctx* x, int use_tensor_cores) {
    if (!x) return fail(MMW_ERR_INVALID, "ctx is NULL");
    x->use_tc = use_tensor_cores != 0;
    return MMW_OK;
}

/* Test hook: the intermediates of the last serial pose-network run (include/mmw.h). */
int mmw_pose_intermediate(mmw_ctx* x, int layer, int* n_rows, void* host_out, size_t bytes) {
    if (!x || !n_rows) return fail(MMW_ERR_INVALID, "ctx/n_rows is NULL");
    if (layer < 0 || layer > 3) return fail(MMW_ERR_INVALID, "layer must be 0..3");
    if (!x->has_weights) return fail(MMW_ERR_STATE, "no pose weights loaded");
    if (x->last_pose_run == 0) return fail(MMW_ERR_STATE, "no pose-network run since the weights were loaded");
    if (x->last_pose_run == 3)
        return fail(MMW_ERR_STATE, "the last pose-network run was in throughput mode (its frame may still be in flight)");
    const bool tc = x->last_pose_run == 1;
    if (!tc && layer < 2) return fail(MMW_ERR_INVALID, "the CUDA-core path keeps layers 2 and 3 only");
    CK(cudaSetDevice(x->device));
    CK(sync_main(x));
    int n = 0;
    CK(cudaMemcpy(&n, x->d_pose_total, sizeof(int), cudaMemcpyDeviceToHost));
    *n_rows = n;
    if (!host_out) return MMW_OK;
    const size_t P = (size_t)x->D * 64;
    const size_t per = layer == 0 ? P * 5 : layer == 1 ? P * 16 : layer == 2 ? (size_t)x->Kf : (size_t)x->H;
    const size_t need = (size_t)n * per * (tc ? 2 * sizeof(uint16_t) : sizeof(float));
    if (bytes < need) return fail(MMW_ERR_CAPACITY, "host_out too small for this layer");
    if (n == 0) return MMW_OK;
    if (tc) {
        if (pose_tc_intermediate(&x->tc, layer, n, static_cast<uint16_t*>(host_out)) != 0)
            return fail(MMW_ERR_CUDA, std::string("pose intermediate: ") + pose_tc_error());
    } else {
        CK(cudaMemcpy(host_out, layer == 2 ? x->d_act2 : x->d_act3, need, cudaMemcpyDeviceToHost));
    }
    return MMW_OK;
}

}  // extern "C"
