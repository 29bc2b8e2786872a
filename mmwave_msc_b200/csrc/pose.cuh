// Argument blocks of the pose-stage kernels (pose_kernels.cu, pose_tc.cu).
#pragma once
#include <cuda_bf16.h>

#include "mmw_internal.cuh"

namespace mmw {

struct PoseFeatArgs {
    DevConfig cfg;
    const SensorRec* sensors;   // [S] each scene's mounting and Doppler unit
    const SceneRec* scenes;
    const TrackRec* tracks;
    const float* track_ring;
    float* feats;          // [rows][ring_size*64*5]
    __nv_bfloat16* packed; // tensor-core conv input [rows][D][8 w][2 chunks: hi|lo][8 h][8 ch] (pose_tc.cu), or nullptr
    int32_t* row_scene;    // [rows]
    int32_t* row_track;
    int32_t* row_slot;
    // Pose-row scan folded into this kernel (pose_cnt != nullptr): CTA s sums pose_cnt[0..s) itself and the CTA of
    // the last scene publishes the row total, so no separate scan kernel sits between the tracker and the features.
    const int32_t* pose_cnt;   // [S] or nullptr (then SceneRec::pose_base from pose_index_kernel is used)
    int* pose_total;
    unsigned long long* counters;
    int n_scenes;
    int dbg = 0;           // timing experiments only (MMW_FEAT_DBG): 1 = no row scan, 2 = no stores, 4 = no rank loop, 8 = no ring loads; 16 = always the exact (float64-order) sort, the fast lattice path off
    const int32_t* late_extra = nullptr;   // non-null: rows only for the tracks step_kernel left (pose_cnt); no wait for
                           //   dbscan_big_kernel except by the thread that publishes pose_total = those rows + *late_extra
    int* rows_hint = nullptr;   // mapped host word that receives the row total (the launcher of dense 1 picks its tile shape from it)
};

struct ConvArgs {
    const float* feats;    // [rows][D*64*5]
    const float *w1, *b1, *w2, *b2, *bn1_scale, *bn1_shift;
    float* act2;           // [rows][D*64*32]  BN1(relu(conv2)), channels-last flatten order
    const int* n_rows;     // device scalar
};

struct FcArgs {
    const float* A;        // [rows][K]
    const float* W;        // [K][H]
    const float *bias, *bn_scale, *bn_shift;
    float* out;            // [rows][H]
    const int* n_rows;
    int K, H;
};

struct Fc2Args {
    const float* act3;     // [rows][H]
    const float* W;        // [H][57]
    const float* bias;
    float* out;            // [rows][57]
    float* keypoints;      // [S][tcap][57] by slot, or nullptr
    const int32_t* row_scene;
    const int32_t* row_slot;
    const int* n_rows;
    int H, tcap;
};

cudaError_t launch_pose_index(SceneRec* scenes, int S, int* pose_total, unsigned long long* counters,
                              cudaStream_t st);
cudaError_t launch_pose_features(const PoseFeatArgs& a, int S, cudaStream_t st);
cudaError_t launch_conv(const ConvArgs& a, int D, int grid, cudaStream_t st);
cudaError_t launch_fc1_simt(const FcArgs& a, int max_rows, cudaStream_t st);
cudaError_t launch_fc2(const Fc2Args& a, int grid, cudaStream_t st);

int step_smem_bytes(int ncap, int tcap);
int dbscan_big_smem_bytes(int ncap);
cudaError_t launch_step(const StepArgs& a, cudaStream_t stream);
cudaError_t launch_dbscan_big(const StepArgs& a, cudaStream_t stream, int grid = 16);

}  // namespace mmw
