// Pose stage: TrackBuffer.estimate_posture (Tracking.py:705-734).
//   pose_index_kernel    compacts the tracks of all scenes that ran this frame into pose rows
//   pose_feature_kernel  relative_coordinates + format_single_frame (Utils.py:437-520) per track
//   conv_kernel          Conv(5->16)+ReLU, Conv(16->32)+ReLU, BatchNorm   (train.py:35-47 / 74-85)
//   fc1 / fc2            Dense+ReLU+BatchNorm, Dense(57)                  (train.py:49-57 / 87-96)
// The CUDA-core fp32 kernels in this file are the reference-exact path; the tensor-core (tcgen05) GEMM for the
// dense contraction lives in pose_tc.cu and replaces fc1 when enabled.
#include "mmw_internal.cuh"
#include <cstdlib>

#include "pose.cuh"
#include "pose_feat.cuh"

namespace mmw {

// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) pose_index_kernel(SceneRec* scenes, int S, int* pose_total,
                                                          unsigned long long* counters) {
    __shared__ int wsum[32];
    __shared__ int running;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) running = 0;
    __syncthreads();
    for (int base = 0; base < S; base += 1024) {
        const int s = base + tid;
        int v = 0;
        if (s < S && scenes[s].last_ran) v = scenes[s].n_tracks;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        int before = 0, tot = 0;
        for (int w = 0; w < 32; ++w) {
            const int cw = wsum[w];
            if (w < warp) before += cw;
            tot += cw;
        }
        const int r0 = running;
        if (s < S) scenes[s].pose_base = r0 + before + incl - v;
        __syncthreads();
        if (tid == 0) running = r0 + tot;
        __syncthreads();
    }
    if (tid == 0) {
        *pose_total = running;
        atomicAdd(&counters[7], (unsigned long long)running);
    }
}

// ---------------------------------------------------------------------------------------------------
// One warp per (track, ring frame): the 3 frames of a track are independent, so a scene with two tracks keeps six
// warps busy at once instead of two warps walking three frames each (round 1: 21 us of dependent round trips for
// 27 MB of traffic).  Feature rows are relative to the CURRENT centroid for every ring frame (Q21), intensity is
// normalised before padding so pads stay exactly 0, rows are sorted by x with the canonical stable (x, row index)
// order, frames absent from the ring stay zero.  Each lane owns points lane and lane + 32 of the frame: their values
// stay in registers, only the 64 sort keys go through shared memory, and both ranks come out of one pass over them.
constexpr int kFeatWarps = 6;
__global__ void __launch_bounds__(kFeatWarps * 32, 7) pose_feature_kernel(PoseFeatArgs a) {
    __shared__ __align__(16) long long keys[kFeatWarps][kFeatPts];     // order-preserving integer images of the sort keys
    __shared__ __align__(16) float srow[kFeatWarps][kFeatPts * kRawCols];
    __shared__ __align__(16) uint4 spk[kFeatWarps][kFeatPts * 2];
    const int s = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // late mode (fused steps): this grid was launched by dbscan_big_kernel's launch_dependents, which that kernel
    // issues after ITS wait for step_kernel -- so step_kernel's results are complete and visible here, and nothing this
    // kernel reads is written by dbscan_big_kernel (it only appends track records and rows).  No wait at the top: the
    // two kernels run side by side.
    const bool late = a.late_extra != nullptr && a.pose_cnt != nullptr;
    if (!late) pdl_wait();               // the tracker kernels have completed
    pdl_launch_dependents();
    SceneRec sc;
    if (!late) sc = a.scenes[s];
    int pose_base = late ? 0 : sc.pose_base;
    int n_tr = 0;
    if (a.dbg & 1) { pose_base = 2 * s; n_tr = late ? __ldg(a.pose_cnt + s) : (sc.last_ran ? sc.n_tracks : 0); }
    else if (a.pose_cnt != nullptr) {
        // exclusive scan value of this scene: every CTA adds up the (at most S) counts in front of it; the order of
        // the integer additions does not matter, so the row layout is the same as pose_index_kernel's
        __shared__ int wpart[kFeatWarps];
        int part = 0;
        for (int i = threadIdx.x; i < s; i += kFeatWarps * 32) part += __ldg(a.pose_cnt + i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) wpart[warp] = part;
        __syncthreads();
        pose_base = 0;
#pragma unroll
        for (int w = 0; w < kFeatWarps; ++w) pose_base += wpart[w];
        n_tr = late ? __ldg(a.pose_cnt + s) : (sc.last_ran ? sc.n_tracks : 0);
    } else {
        n_tr = sc.last_ran ? sc.n_tracks : 0;
    }
    const DevConfig& c = a.cfg;
    __shared__ SensorRec sr;             // the scene's mounting and Doppler unit
    if (threadIdx.x < sizeof(SensorRec) / 8)
        reinterpret_cast<double*>(&sr)[threadIdx.x] = reinterpret_cast<const double*>(a.sensors + s)[threadIdx.x];
    __syncthreads();
    const int nfr = c.ring_size;
    const int items = n_tr * nfr;
    for (int item = warp; item < items; item += kFeatWarps) {
        const int k = item / nfr, f = item - k * nfr;
        const TrackRec* t = a.tracks + (size_t)s * c.tcap + k;
        const int row = pose_base + k;
        const int slot = t->slot, rn = t->ring_n, rh = t->ring_head;
        if (f == 0 && lane == 0) {
            a.row_scene[row] = s;
            a.row_track[row] = k;
            a.row_slot[row] = slot;
        }
        float* out = a.feats + ((size_t)row * nfr + f) * (kFeatPts * kRawCols);
        uint4* pk = a.packed ? reinterpret_cast<uint4*>(a.packed + (size_t)row * nfr * kFeatPts * 16) : nullptr;
        const float* src = nullptr;
        int cnt = 0;
        if (f < rn) {
            const int phys = ring_wrap(rh + f, c.ring_size);
            cnt = t->ring_cnt[phys];
            src = a.track_ring + (((size_t)s * c.tcap + slot) * kRing + phys) * (kFeatPts * kRawCols);
        }
        pose_feature_item<true>(c, sr, src, cnt, t->centroid[0], t->centroid[1], f, out, pk, keys[warp], srow[warp],
                                spk[warp], lane, a.dbg);
    }
    if (a.pose_cnt != nullptr && !(a.dbg & 1) && s == a.n_scenes - 1 && threadIdx.x == 0) {
        int total = pose_base + n_tr;
        if (late) {
            pdl_wait();                  // dbscan_big_kernel has completed: the rows it appended are counted and written
            total += __ldcg(a.late_extra);
        }
        *a.pose_total = total;
        if (a.rows_hint != nullptr) *a.rows_hint = total;            // zero-copy write to pinned host memory
        atomicAdd(&a.counters[7], (unsigned long long)total);
    }
}

// ---------------------------------------------------------------------------------------------------
// Conv stack, one CTA per pose row.  D = 1 (define_CNN, 8x8x5) or 3 (define_CNN_3D, 3x8x8x5).
// 'same' zero padding, cross-correlation, channels-last; Dropout is identity at inference.
template <int D>
__global__ void __launch_bounds__(256) conv_kernel(ConvArgs a) {
    constexpr int P = D * 64;                 // output positions
    constexpr int TAPS = (D == 3 ? 27 : 9);
    constexpr int A1S = 17;                   // padded row stride of act1 (bank conflicts)
    extern __shared__ __align__(16) float sm[];
    float* w2 = sm;                           // [TAPS][16][32]
    float* w1 = w2 + TAPS * 16 * 32;          // [TAPS][5][16]
    float* in = w1 + TAPS * 5 * 16;           // [P][5]
    float* a1 = in + P * 5;                   // [P][A1S]
    __shared__ int total;
    if (threadIdx.x == 0) total = *a.n_rows;
    for (int i = threadIdx.x; i < TAPS * 16 * 32; i += 256) w2[i] = a.w2[i];
    for (int i = threadIdx.x; i < TAPS * 5 * 16; i += 256) w1[i] = a.w1[i];
    __syncthreads();
    for (int row = blockIdx.x; row < total; row += gridDim.x) {
        const float* feat = a.feats + (size_t)row * P * 5;
        for (int i = threadIdx.x; i < P * 5; i += 256) in[i] = feat[i];
        __syncthreads();
        // conv1: thread = (pos, 8 output channels)
        for (int it = threadIdx.x; it < P * 2; it += 256) {
            const int pos = it >> 1, c0 = (it & 1) * 8;
            const int d = pos / 64, h = (pos / 8) % 8, w = pos % 8;
            float acc[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[q] = a.b1[c0 + q];
            for (int tap = 0; tap < TAPS; ++tap) {
                const int kd = (D == 3) ? tap / 9 - 1 : 0, kh = (tap / 3) % 3 - 1, kw = tap % 3 - 1;
                const int dd = d + kd, hh = h + kh, ww = w + kw;
                if (dd < 0 || dd >= D || hh < 0 || hh >= 8 || ww < 0 || ww >= 8) continue;
                const float* ip = in + ((dd * 8 + hh) * 8 + ww) * 5;
                const float* wp_ = w1 + tap * 5 * 16 + c0;
#pragma unroll
                for (int ci = 0; ci < 5; ++ci) {
                    const float v = ip[ci];
#pragma unroll
                    for (int q = 0; q < 8; ++q) acc[q] = fmaf(v, wp_[ci * 16 + q], acc[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) a1[pos * A1S + c0 + q] = fmaxf(acc[q], 0.f);
        }
        __syncthreads();
        // conv2 + ReLU + BatchNorm: thread = (pos, 8 output channels)
        float* out = a.act2 + (size_t)row * P * 32;
        for (int it = threadIdx.x; it < P * 4; it += 256) {
            const int pos = it % P, c0 = (it / P) * 8;
            const int d = pos / 64, h = (pos / 8) % 8, w = pos % 8;
            float acc[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) acc[q] = a.b2[c0 + q];
            for (int tap = 0; tap < TAPS; ++tap) {
                const int kd = (D == 3) ? tap / 9 - 1 : 0, kh = (tap / 3) % 3 - 1, kw = tap % 3 - 1;
                const int dd = d + kd, hh = h + kh, ww = w + kw;
                if (dd < 0 || dd >= D || hh < 0 || hh >= 8 || ww < 0 || ww >= 8) continue;
                const float* ip = a1 + ((dd * 8 + hh) * 8 + ww) * A1S;
                const float* wp_ = w2 + tap * 16 * 32 + c0;
#pragma unroll
                for (int ci = 0; ci < 16; ++ci) {
                    const float v = ip[ci];
#pragma unroll
                    for (int q = 0; q < 8; ++q) acc[q] = fmaf(v, wp_[ci * 32 + q], acc[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
                out[pos * 32 + c0 + q] = fmaf(fmaxf(acc[q], 0.f), a.bn1_scale[c0 + q], a.bn1_shift[c0 + q]);
        }
        __syncthreads();
    }
}

size_t conv_smem_bytes(int D) {
    const int P = D * 64, TAPS = (D == 3 ? 27 : 9);
    return sizeof(float) * (size_t)(TAPS * 16 * 32 + TAPS * 5 * 16 + P * 5 + P * 17);
}

cudaError_t launch_conv(const ConvArgs& a, int D, int grid, cudaStream_t st) {
    const size_t smem = conv_smem_bytes(D);
    cudaError_t e;
    if (D == 3) {
        e = cudaFuncSetAttribute(conv_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        conv_kernel<3><<<grid, 256, smem, st>>>(a);
    } else {
        e = cudaFuncSetAttribute(conv_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        conv_kernel<1><<<grid, 256, smem, st>>>(a);
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------
// Dense 1 (CUDA-core fp32 path): out[n][H] = BN2(relu(A[n][K] W[K][H] + b)).  64x64 tile, 256 threads, 4x4 each.
__global__ void __launch_bounds__(256) fc1_simt_kernel(FcArgs a) {
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int n = *a.n_rows;
    const int m0 = blockIdx.y * 64, h0 = blockIdx.x * 64;
    if (m0 >= n) return;
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < a.K; k0 += 16) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            const int r = i / 16, kk = i % 16;
            As[kk][r] = (m0 + r < n) ? a.A[(size_t)(m0 + r) * a.K + k0 + kk] : 0.f;
        }
        for (int i = threadIdx.x; i < 16 * 64; i += 256) {
            const int kk = i / 64, cc = i % 64;
            Bs[kk][cc] = a.W[(size_t)(k0 + kk) * a.H + h0 + cc];
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float av[4], bv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= n) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int h = h0 + tx * 4 + j;
            const float v = fmaxf(acc[i][j] + a.bias[h], 0.f);
            a.out[(size_t)m * a.H + h] = fmaf(v, a.bn_scale[h], a.bn_shift[h]);
        }
    }
}

cudaError_t launch_fc1_simt(const FcArgs& a, int max_rows, cudaStream_t st) {
    dim3 grid(a.H / 64, (max_rows + 63) / 64);
    fc1_simt_kernel<<<grid, 256, 0, st>>>(a);
    return cudaGetLastError();
}

// Dense 2: keypoints[n][57] = act3[n][H] W3[H][57] + b3.  One CTA = 8 rows; thread = (output o, K half); the
// weight element is loaded once and used for the 8 rows staged in shared memory.  Also scatters the result to the
// owning track's keypoint slot (Tracking.py:733-734).
constexpr int kFc2Rows = 8;
__global__ void __launch_bounds__(128) fc2_kernel(Fc2Args a) {
    extern __shared__ float xs[];                 // [kFc2Rows][H]
    __shared__ float part[kFc2Rows][64];
    const int n = *a.n_rows;
    const int o = threadIdx.x & 63, half = threadIdx.x >> 6;
    const int hlen = a.H / 2;
    for (int r0 = blockIdx.x * kFc2Rows; r0 < n; r0 += gridDim.x * kFc2Rows) {
        const int nr = min(kFc2Rows, n - r0);
        for (int i = threadIdx.x; i < kFc2Rows * a.H; i += 128) {
            const int r = i / a.H;
            xs[i] = r < nr ? a.act3[(size_t)(r0 + r) * a.H + (i - r * a.H)] : 0.f;
        }
        __syncthreads();
        float acc[kFc2Rows];
#pragma unroll
        for (int r = 0; r < kFc2Rows; ++r) acc[r] = 0.f;
        if (o < kKp) {
            const float* wp_ = a.W + (size_t)(half * hlen) * kKp + o;
            const float* xp = xs + half * hlen;
#pragma unroll 4
            for (int h = 0; h < hlen; ++h) {
                const float w = __ldg(wp_ + (size_t)h * kKp);
#pragma unroll
                for (int r = 0; r < kFc2Rows; ++r) acc[r] = fmaf(xp[r * a.H + h], w, acc[r]);
            }
        }
        if (half == 1) {
#pragma unroll
            for (int r = 0; r < kFc2Rows; ++r) part[r][o] = acc[r];
        }
        __syncthreads();
        if (half == 0 && o < kKp) {
#pragma unroll
            for (int r = 0; r < kFc2Rows; ++r) {
                if (r >= nr) break;
                const float v = (acc[r] + part[r][o]) + a.bias[o];
                const int row = r0 + r;
                a.out[(size_t)row * kKp + o] = v;
                if (a.keypoints != nullptr) {
                    const int s = a.row_scene[row], slot = a.row_slot[row];
                    a.keypoints[((size_t)s * a.tcap + slot) * kKp + o] = v;
                }
            }
        }
        __syncthreads();
    }
}

cudaError_t launch_fc2(const Fc2Args& a, int grid, cudaStream_t st) {
    const size_t smem = (size_t)kFc2Rows * a.H * sizeof(float);
    static int configured[kMaxDevices] = {0};
    cudaError_t e = ensure_smem_attr(reinterpret_cast<const void*>(fc2_kernel), configured, 64 * 1024);
    if (e != cudaSuccess) return e;
    fc2_kernel<<<grid, 128, smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pose_index(SceneRec* scenes, int S, int* pose_total, unsigned long long* counters,
                              cudaStream_t st) {
    pose_index_kernel<<<1, 1024, 0, st>>>(scenes, S, pose_total, counters);
    return cudaGetLastError();
}

cudaError_t launch_pose_features(const PoseFeatArgs& a, int S, cudaStream_t st) {
    static int configured[kMaxDevices] = {0};   // same shared-memory carve-out as its neighbours in the step
    cudaError_t e = ensure_smem_attr(reinterpret_cast<const void*>(pose_feature_kernel), configured, -1);
    if (e != cudaSuccess) return e;
    const char* env = getenv("MMW_FEAT_DBG");              // read at every launch: a test switches paths in one process
    const int dbg = env ? atoi(env) : 0;
    PoseFeatArgs b = a;
    b.dbg = dbg;
    return launch_pdl(pose_feature_kernel, dim3(S), dim3(kFeatWarps * 32), 0, st, dim3(1, 1, 1), b);
}

}  // namespace mmw
