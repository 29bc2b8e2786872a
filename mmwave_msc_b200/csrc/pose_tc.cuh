// Tensor-core (tcgen05 + TMEM + TMA) path of the pose network: both convolutions as TMA-im2col implicit GEMMs
// and both dense layers as split-bf16 GEMMs.  See pose_tc.cu for the design notes.
#pragma once
#include <cuda_bf16.h>

#include "pose.cuh"

namespace mmw {

struct PoseTc {
    bool ready = false;
    int D = 0, K = 0, H = 0, rows_cap = 0;
    void* impl = nullptr;
};

struct PoseTcRun {
    const int* n_rows;                 // device scalar: pose rows of this batch
    const float *b1, *b2, *bn1_scale, *bn1_shift, *bd1, *bn2_scale, *bn2_shift, *bd2;
    float* out;                        // [rows][57]
    float* keypoints;                  // [S][tcap][57] by slot or nullptr
    const int32_t *row_scene, *row_slot;
    int tcap;
    // throughput mode (MMW_STEP_PIPELINE): dense 2 also finishes the packed result records of the rows' tracks --
    // keypoints and fade square into results[(scene * tcap + row_track) * 72 + ...] -- so that no kernel of this
    // frame has to read the track records after the next frame's tracker has started on them
    float* results = nullptr;
    const int32_t* row_track = nullptr;
    FadeCfg fade = {0, 0, 0, 0, 0, 0};
};

// host_blob: Keras get_weights() blob, off[i] = float offset of array i (16 arrays).
int pose_tc_init(PoseTc* tc, const float* host_blob, const size_t* off, int D, int rows_cap);
// Packed network input the feature kernel writes: [rows][D][8][8][16] bf16 = (hi c0..4, 0 0 0 | lo c0..4, 0 0 0).
__nv_bfloat16* pose_tc_input(PoseTc* tc, int buf = 0);   // buf 0 / 1: the two input buffers of the throughput mode
// fp32 feature maps [rows][D*64][5] -> packed input (used by the stage-level mmw_pose entry point).
int pose_tc_pack_input(PoseTc* tc, const float* feats, const int* n_rows, cudaStream_t st);
int pose_tc_conv(PoseTc* tc, const PoseTcRun& r, cudaStream_t st, int* n_launches, int buf = 0);
// rows_hint: row count of an earlier frame (0 = unknown): picks 256 x 176, 256 x 192 or 256 x 256 tiles, whichever
// costs the least waves of CTA pairs times tile width -- speed only, the three kernels give the same bits
int pose_tc_fc1(PoseTc* tc, const PoseTcRun& r, int max_rows, cudaStream_t st, int* n_launches, int rows_hint = 0);
int pose_tc_fc2(PoseTc* tc, const PoseTcRun& r, int max_rows, cudaStream_t st, int* n_launches);
// Test hook: layer 0..3 of the last run on input buffer 0, rows [0, n), positions in Keras order (d, h, w, c), as two
// planes (bf16 hi bits, then lo bits) of n * per-row values each (mmw_pose_intermediate).  Synchronous.
int pose_tc_intermediate(PoseTc* tc, int layer, int n, uint16_t* out);
void pose_tc_free(PoseTc* tc);
const char* pose_tc_error();

}  // namespace mmw
