// The fused per-frame tracker step: one CTA of 128 threads per scene runs
//   Utils.normalize_data (Utils.py:342-434) -> TrackBuffer.track (Tracking.py:664-703)
// i.e. transform + bounds filter + ordered compaction, Kalman predict, Mahalanobis gating and association, per-track
// cluster statistics and ring push, track maintenance, Kalman update, push of the unassigned points into the scene's
// global ring and the grid screen that decides whether DBSCAN has anything to find -- with every intermediate in
// shared memory / registers.  HBM traffic per scene-frame is the raw points in, the track records in and out, the
// ring rows written and three 272-byte cell histograms for the screen.
//
// How the work is laid out (round 2; profiles/r02_*.md):
//   * inputs arrive by four bulk copies (cp.async.bulk, 1-D TMA) behind one mbarrier: the scene's contiguous block
//     of raw points (as the 16-byte aligned window around it), its track records, the ring's cell histograms and the
//     scene's sensor record (mounting, Doppler unit, Q format; read from shared memory where it is used);
//   * point phases are thread-per-point, two points per thread per tile of 256, both in flight at once (straight-
//     line code, two independent float64 chains) -- transform, filter, gate, list positions, ring pushes all work
//     from registers;
//   * track phases are ELEMENT-parallel (linalg.cuh): thread e owns element e of the 9x9 / 9x6 / 6x6 matrices and
//     the CTA walks the tracks, so all four warps work whatever the number of tracks; the two 6x6 inverses per
//     track run two tracks per warp (one half warp each);
//   * per-track statistics are a Gram matrix: each associated point leaves the row (d0..d5, x) with d = w - H x in
//     shared memory, in list order, and one warp per track accumulates [1 d x]' [1 d x] over four points per
//     DMMA.8x8x4 (float64 tensor-core MMA; fixed summation order, deterministic) -- sums, second moments and the
//     exact sum of the x lattice values in 1/4 instruction per point; minima / maxima by a second warp;
//   * the grid screen works on per-frame cell histograms that were filled when the frames were pushed; clusters
//     that form are left to dbscan_big_kernel through a work list.
#include "dbscan.cuh"
#include "linalg.cuh"
#include "mmw_internal.cuh"
#include "pose_feat.cuh"

namespace mmw {

constexpr int kTile = 2 * kStepThreads;          // points per tile: two per thread
constexpr int kChunks = kTile / 32;              // warp chunks of 32 consecutive points in a tile
constexpr int kLw = 7;                           // doubles per list row: d0..d5 (w - H x of the point's track), x
constexpr int kBw = 72;                          // doubles of per-track scratch B
// inside B from the gate matrices to the association results: gate form (kGateWords = 28) | new N_est | minima of
// d (6) | maxima of d (6) | sum d (6), sum x, products d_r d_c (21)
constexpr int kGp = 0, kHx = kGp + 21, kNest = 28, kMin = 29, kMax = 35, kSum = 41, kSumX = 47, kProd = 48;
static_assert(kProd + 21 <= kBw, "B holds the statistics totals next to the gate form");
static_assert(kStepThreads == 128, "the element-parallel track phases are written for 128 threads per scene");

// Dynamic shared memory of step_kernel.
//   sensor  the scene's SensorRec (48 bytes; first, so that its address is a constant)
//   tracks  TrackRec [tcap]
//   B       double [tcap][72]   gate..association: see above;  update: S -> S^-1 (0..35) | Rc (36..71)
//   A       double [tcap][81]   F P (predict), C (gate matrix, first 36), (I - K H) P (update)
//   KK      double [tcap][108]  K (0..53) | K Rc (54..107)
//   hist    ring frames' cell histograms (3 x 272 bytes), this frame's counts (256 x uint16)
//   aliases: the list rows of a tile's associated points (kTile x 7 doubles) lie over A|KK between the gate matrices
//   and the update; the staged raw points lie over KK when a frame is a single tile, in their own space otherwise
//   (they must survive the tile loop).
struct SmemLayout {
    int sensor, tracks, B, A, KK, stage, hist, hnew, misc, total;
};
constexpr int kMiscInts = 192;
// misc int slots (slot 0-1: the mbarrier)
enum { kT1 = 2, kFreed = 3, kFlag = 4, kCntK = 8 /* 8 */, kCntU = 16 /* 8 */, kBaseG = 24 /* 2 x 32 */,
       kBaseU = 88 /* 2 */, kOrder = 92 /* 32 */, kCntG = 124 /* 8 x 32 bytes = 64 ints */ };
static_assert(kCntG + 64 <= kMiscInts, "misc layout");

__host__ __device__ inline SmemLayout make_layout(int ncap, int tcap) {
    SmemLayout L;
    int o = 0;
    L.sensor = o;  o += (int)sizeof(SensorRec);
    L.tracks = o;  o += tcap * (int)sizeof(TrackRec);
    L.B = o;       o += tcap * kBw * 8;
    L.A = o;
    const int a_bytes = (tcap * 81 * 8 + 15) & ~15;      // KK (bulk-copy destination when it stages the points) stays 16-byte aligned
    int kk_bytes = tcap * 108 * 8;
    const int stage_bytes = ((ncap * kRawCols * 4 + 15) & ~15) + 32;
    const bool single = ncap <= kTile;
    if (single && kk_bytes < stage_bytes) kk_bytes = stage_bytes;
    int akk = a_bytes + kk_bytes;
    const int list_bytes = kTile * kLw * 8;
    if (akk < list_bytes) akk = list_bytes;
    akk = (akk + 15) & ~15;
    L.KK = L.A + a_bytes;
    o += akk;
    L.stage = single ? L.KK : o;
    if (!single) o += stage_bytes;
    L.hist = o;    o += kRing * kHistBytes;
    L.hnew = o;    o += kGridCells * 2;
    L.misc = o;    o += kMiscInts * 4;
    L.total = o;
    return L;
}

int step_smem_bytes(int ncap, int tcap) { return make_layout(ncap, tcap).total; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// ---- mbarrier + bulk copy (1-D TMA) ------------------------------------------------------------------
__device__ __forceinline__ uint32_t sk_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sk_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sk_smem(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void sk_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sk_smem(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sk_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "SK_WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra SK_DONE;\n\t"
        "bra SK_WAIT_LOOP;\n\t"
        "SK_DONE:\n\t"
        "}" ::"r"(sk_smem(bar)), "r"(parity) : "memory");
}
// bytes: a positive multiple of 16; dst (shared) and src (global) 16-byte aligned
__device__ __forceinline__ void sk_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
                     "r"(sk_smem(dst)), "l"(src), "r"(bytes), "r"(sk_smem(bar))
                 : "memory");
}
// D (8x8, float64) += A (8x4) B (4x8): lane L supplies A[L/4][L%4] and B[L%4][L/4], holds D[L/4][2 (L%4) + {0, 1}]
__device__ __forceinline__ void dmma_884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ const float* uring_frame(const StepArgs& a, int s, int phys) {
    return a.uring + ((size_t)s * kRing + phys) * (size_t)a.cfg.ncap * kRawCols;
}

// One warp turns DBSCAN cluster q of the fused ring into a fresh track (ClusterTrack.__init__, Tracking.py:210-230
// over PointCluster(cluster), :120-136): statistics over the 6 world columns recomputed from the ring's raw rows,
// state x = [centroid, 0, 0, 0], P = KF_P_INIT*I, group dispersion = KF_GROUP_DISP_EST_INIT*I, ring = [first 64
// cluster rows in fused order], keypoints = MODEL_DEFAULT_POSTURE.  `t` may live in shared or global memory.
__device__ __forceinline__ void spawn_track(const StepArgs& a, const SensorRec& sr, int s, TrackRec& t, int q, int slot,
                                            int track_id, const int* cl, const int* fcnt, const int* fphys, int lane,
                                            const float* rawc = nullptr /* fused raw rows in shared memory */,
                                            const double* w6 = nullptr /* their world 6-vectors, precomputed */) {
    const DevConfig& c = a.cfg;
    const int tcap = c.tcap;
    int n = 0;
    double sacc[6], mn[6], mx[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) { sacc[k] = 0.0; mn[k] = INFINITY; mx[k] = -INFINITY; }
    int b0 = 0;
    float* dst = a.track_ring + (((size_t)s * tcap + slot) * kRing + 0) * (kFeatPts * kRawCols);
    int stored = 0;
    for (int f = 0; f < kRing; ++f) {
        const float* src = rawc != nullptr ? rawc + (size_t)b0 * kRawCols : uring_frame(a, s, fphys[f]);
        for (int i0 = 0; i0 < fcnt[f]; i0 += 32) {
            const int i = i0 + lane;
            const bool in = i < fcnt[f] && cl[b0 + i] == q;
            float r5[kRawCols];
            if (in) {
#pragma unroll
                for (int k = 0; k < kRawCols; ++k) r5[k] = src[i * kRawCols + k];
                double w[6];
                if (w6 != nullptr) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) w[k] = w6[(size_t)(b0 + i) * 6 + k];
                } else {
                    world_from_raw(sr, r5[0], r5[1], r5[2], r5[3], w);
                }
                ++n;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    sacc[k] += w[k]; mn[k] = fmin(mn[k], w[k]); mx[k] = fmax(mx[k], w[k]);
                }
            }
            const unsigned m = __ballot_sync(kFull, in);
            const int pos = stored + __popc(m & ((1u << lane) - 1u));
            if (in && pos < kFeatPts) {
#pragma unroll
                for (int k = 0; k < kRawCols; ++k) dst[pos * kRawCols + k] = r5[k];
            }
            stored += __popc(m);
        }
        b0 += fcnt[f];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(kFull, n, o);
    double cen[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        cen[k] = warp_sum(sacc[k]) / (double)n;
        mn[k] = warp_min(mn[k]);
        mx[k] = warp_max(mx[k]);
    }
    for (int e = lane; e < 81; e += 32) t.P[e] = (e / 9 == e % 9) ? c.p_init : 0.0;
    for (int e = lane; e < 36; e += 32) t.G[e] = (e / 6 == e % 6) ? c.g_init : 0.0;
    if (lane >= 6 && lane < 9) t.x[lane] = 0.0;
    if (lane < 6) {
        t.x[lane] = cen[lane];
        t.centroid[lane] = cen[lane];
        t.minv[lane] = mn[lane];
        t.maxv[lane] = mx[lane];
        t.spread[lane] = 0.0;
    }
    if (lane == 0) {
        t.n_est = 0.0;
        t.lifetime = 0.0;
        t.id = track_id;
        t.point_num = n;
        t.is_static = sqrt(cen[3] * cen[3] + cen[4] * cen[4] + cen[5] * cen[5]) < c.vel_thres ? 1 : 0;
        t.slot = slot;
        t.ring_n = 1;
        t.ring_head = 0;
        t.ring_cnt[0] = n < kFeatPts ? n : kFeatPts;
        t.ring_cnt[1] = 0;
        t.ring_cnt[2] = 0;
        t.pad[0] = t.pad[1] = t.pad[2] = 0;
    }
    // keypoints = MODEL_DEFAULT_POSTURE until the first inference (Tracking.py:221, Q25)
    float* kp = a.keypoints + ((size_t)s * tcap + slot) * kKp;
    for (int e = lane; e < kKp; e += 32) kp[e] = a.default_posture[e];
}

// The same for the bit-matrix path of dbscan_big_kernel, by the whole CTA (16 warps) instead of one warp per cluster: the
// cluster's points are spread over all threads (fused clouds of <= 768 points: at most two per thread), sums / minima /
// maxima are reduced per warp by shuffles and across warps in warp order (fixed order: deterministic), the first 64
// cluster rows in fused order get their ring positions from per-chunk ballot counts, and the record's fields are
// written by different threads at once.  `red` is shared scratch of at least 16 * 20 + 32 + 20 doubles.
__device__ __forceinline__ void spawn_track_block(const StepArgs& a, int s, TrackRec& t, int q, int slot, int track_id,
                                                  const int* cl, int B, const float* rawc, const double* w6, double* red) {
    const DevConfig& c = a.cfg;
    const int tcap = c.tcap, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const unsigned ltmask = (1u << lane) - 1u;
    double* wred = red;                                   // [nwarps][20]: n, sums (6), minima (6), maxima (6)
    int* ccnt = reinterpret_cast<int*>(red + nwarps * 20);   // [<= 32] in-cluster points per chunk of 32
    double* fin = red + nwarps * 20 + 16;                 // [20] totals
    const int nchunks = (B + 31) >> 5;
    int n = 0;
    double sacc[6], mn[6], mx[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) { sacc[k] = 0.0; mn[k] = INFINITY; mx[k] = -INFINITY; }
    unsigned mask[2] = {0u, 0u};
    for (int j = 0, ch = warp; ch < nchunks; ch += nwarps, ++j) {
        const int b = ch * 32 + lane;
        const bool in = b < B && cl[b] == q;
        if (in) {
            ++n;
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                const double w = w6[(size_t)b * 6 + k];
                sacc[k] += w; mn[k] = fmin(mn[k], w); mx[k] = fmax(mx[k], w);
            }
        }
        const unsigned m = __ballot_sync(kFull, in);
        if (j < 2) mask[j] = m;
        if (lane == 0) ccnt[ch] = __popc(m);
    }
    if (__any_sync(kFull, n > 0)) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(kFull, n, o);
#pragma unroll
        for (int k = 0; k < 6; ++k) { sacc[k] = warp_sum(sacc[k]); mn[k] = warp_min(mn[k]); mx[k] = warp_max(mx[k]); }
    }
    if (lane == 0) {
        double* w = wred + warp * 20;
        w[0] = (double)n;
#pragma unroll
        for (int k = 0; k < 6; ++k) { w[1 + k] = sacc[k]; w[7 + k] = mn[k]; w[13 + k] = mx[k]; }
    }
    __syncthreads();
    if (warp == 0 && lane < 19) {                        // across the warps, in warp order
        double v = wred[lane];
        for (int w = 1; w < nwarps; ++w) {
            const double o = wred[w * 20 + lane];
            v = lane < 7 ? v + o : (lane < 13 ? fmin(v, o) : fmax(v, o));
        }
        fin[lane] = v;
    }
    // ring = the first 64 cluster rows in fused order (ClusterTrack.__init__ -> BatchedData of the cluster's points)
    float* dst = a.track_ring + (((size_t)s * tcap + slot) * kRing + 0) * (kFeatPts * kRawCols);
    for (int j = 0, ch = warp; ch < nchunks && j < 2; ch += nwarps, ++j) {
        const int b = ch * 32 + lane;
        if ((mask[j] >> lane) & 1u) {
            int before = 0;
            for (int c2 = 0; c2 < ch; ++c2) before += ccnt[c2];
            const int pos = before + __popc(mask[j] & ltmask);
            if (pos < kFeatPts) {
#pragma unroll
                for (int k = 0; k < kRawCols; ++k) dst[pos * kRawCols + k] = rawc[(size_t)b * kRawCols + k];
            }
        }
    }
    __syncthreads();
    const int ntot = (int)fin[0];
    const double cen = tid < 6 ? fin[1 + tid] / (double)ntot : 0.0;
    if (tid < 81) t.P[tid] = (tid / 9 == tid % 9) ? c.p_init : 0.0;
    else if (tid >= 96 && tid < 132) { const int e = tid - 96; t.G[e] = (e / 6 == e % 6) ? c.g_init : 0.0; }
    else if (tid >= 160 && tid < 163) t.x[6 + tid - 160] = 0.0;
    else if (tid >= 192 && tid < 192 + kKp)               // keypoints = MODEL_DEFAULT_POSTURE until the first inference (Q25)
        a.keypoints[((size_t)s * tcap + slot) * kKp + (tid - 192)] = a.default_posture[tid - 192];
    if (tid < 6) {
        t.x[tid] = cen;
        t.centroid[tid] = cen;
        t.minv[tid] = fin[7 + tid];
        t.maxv[tid] = fin[13 + tid];
        t.spread[tid] = 0.0;
    }
    if (tid == 32) {
        const double c3 = fin[4] / (double)ntot, c4 = fin[5] / (double)ntot, c5 = fin[6] / (double)ntot;
        t.n_est = 0.0;
        t.lifetime = 0.0;
        t.id = track_id;
        t.point_num = ntot;
        t.is_static = sqrt(c3 * c3 + c4 * c4 + c5 * c5) < c.vel_thres ? 1 : 0;
        t.slot = slot;
        t.ring_n = 1;
        t.ring_head = 0;
        t.ring_cnt[0] = ntot < kFeatPts ? ntot : kFeatPts;
        t.ring_cnt[1] = 0;
        t.ring_cnt[2] = 0;
        t.pad[0] = t.pad[1] = t.pad[2] = 0;
    }
    __syncthreads();                     // `red` is reused by the next cluster
}

// fp32 world coordinates of the fused ring (oldest frame first) into shared memory + the screened predicate over
// them (dbscan.cuh).  Block-cooperative; ends with __syncthreads().
__device__ __forceinline__ NbScreened load_fused_ring(const StepArgs& a, const SensorRec& sr, int s, const int* fcnt,
                                                      const int* fphys, float* Xf, int stride, float* rawc = nullptr) {
    const DevConfig& c = a.cfg;
    float* Yf = Xf + stride;
    float* Zf = Yf + stride;
    NbScreened nb{c, sr, Xf, Yf, Zf, {nullptr, nullptr, nullptr}, {0, 0, 0, 0}, c.db_eps, c.screen_lo, c.screen_hi,
                  (float)c.db_range_weight, (float)c.db_z_weight, rawc};
    static_assert(kRing == 3, "the flattened ring load below is written for three frames");
    int b0 = 0;
    for (int f = 0; f < kRing; ++f) {
        nb.frame[f] = uring_frame(a, s, fphys[f]);
        nb.start[f] = b0;
        b0 += fcnt[f];
    }
    nb.start[kRing] = b0;
    // one pass over the fused cloud: the loads of the three frames are independent (a loop per frame paid three round
    // trips to HBM one after the other)
    for (int b = threadIdx.x; b < b0; b += blockDim.x) {
        const int f = b >= nb.start[2] ? 2 : (b >= nb.start[1] ? 1 : 0);
        const float* src = nb.frame[f];
        const int i = b - nb.start[f];
        const float x = src[i * kRawCols + 0], y = src[i * kRawCols + 1], z = src[i * kRawCols + 2];
        double yw, zw;
        world_yz(sr, (double)y, (double)z, yw, zw);
        Xf[b] = screen_domain_mark(x, yw, zw, c.screen_rmax); Yf[b] = (float)yw; Zf[b] = (float)zw;
        if (rawc != nullptr) {
            float* r = rawc + (size_t)b * kRawCols;
            r[0] = x; r[1] = y; r[2] = z; r[3] = src[i * kRawCols + 3]; r[4] = src[i * kRawCols + 4];
        }
    }
    __syncthreads();
    return nb;
}



// Optional per-phase cycle accounting (thread 0 of every CTA, accumulated with one atomic per phase).
#define PHASE_MARK(idx)                                                                  \
    do {                                                                                 \
        if (dbg_clocks && threadIdx.x == 0) {                                            \
            const long long now__ = clock64();                                           \
            atomicAdd(&a.phase_cycles[idx], (unsigned long long)(now__ - phase_t0));     \
            phase_t0 = now__;                                                            \
        }                                                                                \
    } while (0)

constexpr int kStepMinBlocks = 7;                // resident scene CTAs per SM the register budget is sized for
__global__ void __launch_bounds__(kStepThreads, kStepMinBlocks) step_kernel(const __grid_constant__ StepArgs a) {
    const bool dbg_clocks = a.phase_cycles != nullptr;
    long long phase_t0 = dbg_clocks ? clock64() : 0;
    const long long kernel_t0 = phase_t0;
    if (dbg_clocks && threadIdx.x == 0) {
        unsigned long long ns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
        a.phase_cycles[16 + gridDim.x + blockIdx.x] = ns;
    }
    extern __shared__ __align__(16) unsigned char smem[];
    const DevConfig& c = a.cfg;
    const int ncap = c.ncap, tcap = c.tcap;
    const SmemLayout L = make_layout(ncap, tcap);
    TrackRec* tr = reinterpret_cast<TrackRec*>(smem + L.tracks);
    double* Bm = reinterpret_cast<double*>(smem + L.B);
    double* Am = reinterpret_cast<double*>(smem + L.A);
    double* KKm = reinterpret_cast<double*>(smem + L.KK);
    double* wl = Am;                                            // list rows (alias A | KK)
    uint8_t* hist = smem + L.hist;                              // [kRing][kHistBytes] by physical ring slot
    uint16_t* hnew = reinterpret_cast<uint16_t*>(smem + L.hnew);   // this frame's cell counts, later the fused sums
    int* misc = reinterpret_cast<int*>(smem + L.misc);
    uint8_t* cntG = reinterpret_cast<uint8_t*>(misc + kCntG);   // [kChunks][32] points per chunk and track
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + L.misc);
    const SensorRec& sr = *reinterpret_cast<const SensorRec*>(smem);   // this scene's mounting (L.sensor = 0)

    const int s = blockIdx.x;
    if (s >= a.n_scenes) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (s == 0 && tid == 0 && a.nr_extra != nullptr) *a.nr_extra = 0;      // rows dbscan_big_kernel will append this frame
    const Elem el(tid);
    const unsigned ltmask = (1u << lane) - 1u;

    // ---- 0. round trip one: scene record, offsets, dt; then the four bulk copies -----------------------------
    if (tid == 0) sk_mbar_init(mbar, 1);
    SceneRec sc = a.scenes[s];           // every thread keeps a copy; thread 0 writes it back
    const int off = a.offsets[s];
    int N = a.offsets[s + 1] - off;
    const double dt = a.dt[s];
    if (N < 0) N = 0;
    if (N > ncap) { N = ncap; sc.flags |= MMW_SCENE_POINT_OVERFLOW; }
    const int T0 = sc.n_tracks;
    __syncthreads();                     // the barrier is initialised
    const bool i16 = (a.flags & MMW_STEP_INPUT_I16) != 0;             // the sensor's int16 lattice, 10 bytes per point
    const int row_bytes = i16 ? kRawCols * 2 : kRawCols * 4;
    const size_t byte0 = (size_t)(a.pts_row0 + off) * row_bytes;
    const size_t win0 = byte0 & ~(size_t)15;
    const uint32_t win_bytes = (uint32_t)(((byte0 + (size_t)N * row_bytes + 15) & ~(size_t)15) - win0);
    const bool bulk_pts = (reinterpret_cast<uintptr_t>(a.pts) & 15) == 0;       // else: plain loads (below)
    const unsigned char* stageb = smem + L.stage + (byte0 - win0);
    const float* stagef = reinterpret_cast<const float*>(stageb);
    const int16_t* stageh = reinterpret_cast<const int16_t*>(stageb);
    if (tid == 0) {
        const uint32_t tr_bytes = (uint32_t)T0 * (uint32_t)sizeof(TrackRec);
        sk_mbar_expect_tx(mbar, tr_bytes + (bulk_pts ? win_bytes : 0u) + (uint32_t)(kRing * kHistBytes + sizeof(SensorRec)));
        if (tr_bytes) sk_bulk_g2s(tr, a.tracks + (size_t)s * tcap, tr_bytes, mbar);
        if (bulk_pts && win_bytes)
            sk_bulk_g2s(smem + L.stage, reinterpret_cast<const unsigned char*>(a.pts) + win0, win_bytes, mbar);
        sk_bulk_g2s(hist, a.ring_hist + (size_t)s * (kRing * kHistBytes), kRing * kHistBytes, mbar);
        sk_bulk_g2s(smem + L.sensor, a.sensors + s, (uint32_t)sizeof(SensorRec), mbar);
    }
    if (!bulk_pts) {
        if (i16) {
            int16_t* st = const_cast<int16_t*>(stageh);
            const int16_t* src = reinterpret_cast<const int16_t*>(a.pts) + (size_t)(a.pts_row0 + off) * kRawCols;
            for (int i = tid; i < N * kRawCols; i += kStepThreads) st[i] = src[i];
        } else {
            float* st = const_cast<float*>(stagef);
            for (int i = tid; i < N * kRawCols; i += kStepThreads) st[i] = a.pts[(size_t)(a.pts_row0 + off) * kRawCols + i];
        }
    }
    reinterpret_cast<uint32_t*>(hnew)[tid] = 0u;                 // 256 uint16 counts = 128 words
    if (tid < 32) misc[kBaseG + tid] = 0;
    if (tid == 32) { misc[kBaseU] = 0; misc[kFlag] = 0; }
    sk_mbar_wait(mbar, 0);
    if (!bulk_pts) __syncthreads();
    PHASE_MARK(1);

    // ---- 1. predict (Tracking.py:591-596, Q9) and gate matrices (Tracking.py:545-551) -----------------------
    // Element-parallel, one track at a time: every thread computes its element of F P F' + Q from the old P, one
    // barrier, then the stores: P, x = F x, H x, and the gate matrix C = P[:6,:6] + Rm + G (get_Rm 361-370) into the
    // track's B block.
    for (int j = 0; j < T0; ++j) {
        TrackRec& t = tr[j];
        double pv = 0.0, xv = 0.0;
        const double dte = t.lifetime + dt;
        if (tid < 81) pv = kf_predict_elem(t.P, dte, c.q_var, el);
        if (tid < 9) xv = kf_predict_x(t.x, dte, tid);
        __syncthreads();
        if (tid < 81) {
            t.P[tid] = pv;
            if (el.i9 < 6 && el.j9 < 6) {
                double v = pv;
                if (el.i9 == el.j9) { const double h = t.spread[el.i9] / 2; v += h * h; }
                Bm[j * kBw + kMin + el.i9 * 6 + el.j9] = v + t.G[el.i9 * 6 + el.j9];
            }
        }
        if (tid < 9) t.x[tid] = xv;
        if (tid < 6) Bm[j * kBw + kHx + tid] = xv;
    }
    __syncthreads();
    PHASE_MARK(2);
    // inverse + log|det| of the gate matrices, two tracks per warp, kept in the packed gate form (linalg.cuh).  The
    // half warp then resets the track's statistics totals, which take the place of C.
    for (int j0 = 0; j0 < T0; j0 += 2 * kStepWarps) {
        const int j = j0 + 2 * warp + (lane >> 4);
        const bool live = j < T0;
        if (__ballot_sync(kFull, live) == 0u) continue;
        double r[6];
        const double det = inv6_spd_half(live ? Bm + j * kBw + kMin : nullptr, lane, r);
        __syncwarp();
        if (live) {
            double* bj = Bm + j * kBw;
            gate_pack_half(bj + kGp, r, det, lane);
            for (int v = lane & 15; v < 40; v += 16) bj[kMin + v] = v < 6 ? INFINITY : (v < 12 ? -INFINITY : 0.0);
        }
    }
    __syncthreads();
    PHASE_MARK(3);

    // ---- 2. tiles of 256 points: transform + filter + compaction (Utils.py:379-432), gating + association
    //         (Tracking.py:553-572, Q14), list positions, ring pushes (Tracking.py:691, 338), statistics ------------
    const int uphys = sc.ring_n >= c.ring_size ? sc.ring_head : ring_wrap(sc.ring_head + sc.ring_n, c.ring_size);
    float* udst = const_cast<float*>(uring_frame(a, s, uphys));
    int M = 0;
    const int ntiles = (N + kTile - 1) / kTile;
    for (int tile = 0; tile < ntiles; ++tile) {
        // both points of the thread in straight-line code: two independent float64 chains in flight
        float raw[2][kRawCols];
        double w[2][6];
        bool keep[2];
        unsigned km[2];
#pragma unroll
        for (int r2 = 0; r2 < 2; ++r2) {
            const int i = tile * kTile + r2 * kStepThreads + tid;
            const int ic = i < N ? i : N - 1;                    // lanes past the end redo the last point (discarded)
            if (i16) {                   // value / 2^Q is exact in fp32; the Doppler column is the index
                const int16_t* p = stageh + ic * kRawCols;
                raw[r2][0] = (float)p[0] * sr.xyz_scale; raw[r2][1] = (float)p[1] * sr.xyz_scale;
                raw[r2][2] = (float)p[2] * sr.xyz_scale; raw[r2][3] = (float)p[3]; raw[r2][4] = (float)p[4];
            } else {
#pragma unroll
                for (int k = 0; k < kRawCols; ++k) raw[r2][k] = stagef[ic * kRawCols + k];
            }
            world_from_raw(sr, raw[r2][0], raw[r2][1], raw[r2][2], raw[r2][3], w[r2]);
            keep[r2] = i < N && (w[r2][2] <= sr.z_max) && (w[r2][2] > 0.0) && (w[r2][1] > 0.0);   // Utils.py:423-427
        }
#pragma unroll
        for (int r2 = 0; r2 < 2; ++r2) {
            km[r2] = __ballot_sync(kFull, keep[r2]);
            if (lane == 0) misc[kCntK + r2 * kStepWarps + warp] = __popc(km[r2]);
        }
        __syncthreads();
        PHASE_MARK(4);
        int pos[2], tile_kept = 0;
        {
            int pre0 = 0, pre1 = 0;
#pragma unroll
            for (int c2 = 0; c2 < kChunks; ++c2) {
                const int v = misc[kCntK + c2];
                tile_kept += v;
                if (c2 < warp) pre0 += v;
                if (c2 < kStepWarps + warp) pre1 += v;
            }
            pos[0] = M + pre0 + __popc(km[0] & ltmask);
            pos[1] = M + pre1 + __popc(km[1] & ltmask);
        }
        // gate: d2 = log|det C| + y' C^-1 y < gate, arg-min over the gated tracks, ties -> lower index
        int grp[2];
        {
            double best0 = INFINITY, best1 = INFINITY;
            int bj0 = -1, bj1 = -1;
            if (keep[0])
                for (int j = 0; j < T0; ++j) {
                    const double d0 = gate_score(Bm + j * kBw + kGp, w[0]);
                    if (d0 < c.gate && d0 < best0) { best0 = d0; bj0 = j; }
                }
            if (keep[1])
                for (int j = 0; j < T0; ++j) {
                    const double d1 = gate_score(Bm + j * kBw + kGp, w[1]);
                    if (d1 < c.gate && d1 < best1) { best1 = d1; bj1 = j; }
                }
            grp[0] = keep[0] ? (bj0 < 0 ? T0 : bj0) : 255;
            grp[1] = keep[1] ? (bj1 < 0 ? T0 : bj1) : 255;
            if (keep[0]) a.assoc_out[off + pos[0]] = bj0;
            if (keep[1]) a.assoc_out[off + pos[1]] = bj1;
        }
        // per chunk and group: count (lane j keeps track j's) and this point's rank inside its group
        int rk[2] = {0, 0};
        {
            int cj[2] = {0, 0};
#pragma unroll
            for (int r2 = 0; r2 < 2; ++r2) {
                for (int j = 0; j < T0; ++j) {
                    const unsigned b = __ballot_sync(kFull, grp[r2] == j);
                    if (grp[r2] == j) rk[r2] = __popc(b & ltmask);
                    if (lane == j) cj[r2] = __popc(b);
                }
                const unsigned bu = __ballot_sync(kFull, grp[r2] == T0);
                if (grp[r2] == T0) rk[r2] = __popc(bu & ltmask);
                if (lane < T0) cntG[(r2 * kStepWarps + warp) * 32 + lane] = (uint8_t)cj[r2];
                if (lane == 0) misc[kCntU + r2 * kStepWarps + warp] = __popc(bu);
            }
        }
        __syncthreads();
        PHASE_MARK(5);
        // lane j: points of track j in this tile, where this warp's two chunks start inside its list, the number of
        // points it had before this tile; the tile-local list of track j starts at the exclusive scan over j
        int tot = 0, preg[2] = {0, 0}, base = 0, start;
        {
            if (lane < T0) {
#pragma unroll
                for (int c2 = 0; c2 < kChunks; ++c2) {
                    const int v = cntG[c2 * 32 + lane];
                    tot += v;
                    if (c2 < warp) preg[0] += v;
                    if (c2 < kStepWarps + warp) preg[1] += v;
                }
                base = misc[kBaseG + (tile & 1) * 32 + lane];
            }
            int incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += up;
            }
            start = incl - tot;
        }
        int ubase = misc[kBaseU + (tile & 1)], utot = 0, preu[2] = {0, 0};
#pragma unroll
        for (int c2 = 0; c2 < kChunks; ++c2) {
            const int v = misc[kCntU + c2];
            utot += v;
            if (c2 < warp) preu[0] += v;
            if (c2 < kStepWarps + warp) preu[1] += v;
        }
        if (warp == 0) {                 // running counts for the next tile (double-buffered: others still read these)
            if (lane < T0) misc[kBaseG + ((tile + 1) & 1) * 32 + lane] = base + tot;
            if (lane == 0) misc[kBaseU + ((tile + 1) & 1)] = ubase + utot;
        }
#pragma unroll
        for (int r2 = 0; r2 < 2; ++r2) {
            const int g = grp[r2];
            const int gs = g < T0 ? g : 0;
            const int gb = __shfl_sync(kFull, base, gs), gp0 = __shfl_sync(kFull, preg[r2], gs),
                      gst = __shfl_sync(kFull, start, gs);
            if (g < T0) {
                const int lp = gb + gp0 + rk[r2];                // position in the track's cloud of this frame
                double* row = wl + (gst + gp0 + rk[r2]) * kLw;   // position in the tile's list
                const double* hx = Bm + g * kBw + kHx;
#pragma unroll
                for (int k = 0; k < 6; ++k) row[k] = w[r2][k] - hx[k];
                row[6] = w[r2][0];
                if (lp < kFeatPts) {
                    // first 64 associated rows in input order are what format_single_frame can see
                    const TrackRec& t = tr[g];
                    const int phys = t.ring_n >= c.ring_size ? t.ring_head : ring_wrap(t.ring_head + t.ring_n, c.ring_size);
                    float* dst = a.track_ring + (((size_t)s * tcap + t.slot) * kRing + phys) * (kFeatPts * kRawCols) +
                                 (size_t)lp * kRawCols;
#pragma unroll
                    for (int k = 0; k < kRawCols; ++k) dst[k] = raw[r2][k];
                }
            } else if (g == T0) {
                // BatchedData.add_frame(unassigned): the oldest frame is dropped when the ring is full
                float* dst = udst + (size_t)(ubase + preu[r2] + rk[r2]) * kRawCols;
#pragma unroll
                for (int k = 0; k < kRawCols; ++k) dst[k] = raw[r2][k];
                // the frame's cell histogram for the grid screen (dbscan.cuh)
                const float yw = (float)w[r2][1];
                if (!(yw <= c.grid_ybound)) misc[kFlag] = 1;
                const int cell = grid_cell(c, raw[r2][0], yw);
                atomicAdd(reinterpret_cast<unsigned*>(hnew) + (cell >> 1), (cell & 1) ? 0x10000u : 1u);
            }
        }
        M += tile_kept;
        __syncthreads();
        PHASE_MARK(6);
        // statistics of this tile's lists (PointCluster, Tracking.py:120-136; _get_D 270-290 about H x instead of the
        // centroid: E[d d'] - m m' with d = w - H x and m = mean d, below the gate radius, so nothing cancels).
        // Track j: warp j % 4 accumulates the Gram matrix of the rows [1 d0..d5 x], four points per DMMA, two
        // accumulator chains; warp (j + 2) % 4 takes the minima / maxima.
        for (int j = 0; j < T0; ++j) {
            const int nj = __shfl_sync(kFull, tot, j), st = __shfl_sync(kFull, start, j);
            if (nj == 0) continue;
            const double* rows = wl + st * kLw;
            double* bj = Bm + j * kBw;
            if (warp == (j & 3)) {
                const int pt = lane & 3, comp = lane >> 2;
                double c0a = 0.0, c1a = 0.0, c0b = 0.0, c1b = 0.0;
                for (int g0 = 0; g0 < nj; g0 += 8) {
                    const int k0 = g0 + pt, k1 = g0 + 4 + pt;
                    double va = 0.0, vb = 0.0;
                    if (k0 < nj) va = comp ? rows[k0 * kLw + comp - 1] : 1.0;
                    if (k1 < nj) vb = comp ? rows[k1 * kLw + comp - 1] : 1.0;
                    dmma_884(c0a, c1a, va, va);
                    dmma_884(c0b, c1b, vb, vb);
                }
                const double cv[2] = {c0a + c0b, c1a + c1b};
#pragma unroll
                for (int e2 = 0; e2 < 2; ++e2) {
                    const int col = 2 * pt + e2;                 // Gram[comp][col]; index 0 = the constant, 7 = x
                    int idx = -1;
                    if (comp == 0) { if (col >= 1) idx = kSum + col - 1; }
                    else if (comp <= 6 && col >= comp && col <= 6) {
                        const int r = comp - 1, q = col - 1;
                        idx = kProd + r * 6 - (r * (r - 1)) / 2 + (q - r);
                    }
                    if (idx >= 0) bj[idx] += cv[e2];
                }
            }
            if (warp == ((j + 2) & 3)) {
                const int dim = lane >> 2, q = lane & 3;
                const int col = dim == 0 ? 6 : dim;              // x itself (exact) for dim 0, d_k otherwise
                double mn = INFINITY, mx = -INFINITY;
                if (lane < 24) {
                    for (int k = q; k < nj; k += 4) {
                        const double v = rows[k * kLw + col];
                        mn = v < mn ? v : mn;
                        mx = v > mx ? v : mx;
                    }
                }
#pragma unroll
                for (int o = 1; o <= 2; o <<= 1) {
                    const double omn = __shfl_xor_sync(kFull, mn, o), omx = __shfl_xor_sync(kFull, mx, o);
                    mn = omn < mn ? omn : mn;
                    mx = omx > mx ? omx : mx;
                }
                if (lane < 24 && q == 0) {
                    const double sh = dim == 0 ? 0.0 : bj[kHx + dim];          // back to world coordinates
                    mn += sh; mx += sh;
                    bj[kMin + dim] = mn < bj[kMin + dim] ? mn : bj[kMin + dim];
                    bj[kMax + dim] = mx > bj[kMax + dim] ? mx : bj[kMax + dim];
                }
            }
        }
        __syncthreads();
    }
    for (int i = M + tid; i < N; i += kStepThreads) a.assoc_out[off + i] = -2;

    sc.last_M = M;
    sc.dbscan_n = -1;
    if (M == 0) {                        // offline_main.py:55: the frame is skipped entirely (Q23)
        if (tid == 0) {
            sc.last_ran = 0;
            a.scenes[s] = sc;
            a.pose_cnt[s] = 0;
            int4* st4 = reinterpret_cast<int4*>(a.scene_stats + (size_t)s * 8);
            st4[0] = make_int4(N, 0, 0, 0);
            st4[1] = make_int4(0, 0, 0, 0);
        }
        return;
    }
    sc.last_ran = 1;
    const int U = misc[kBaseU + (ntiles & 1)];
    PHASE_MARK(7);

    // ---- 3. per-track association results (Tracking.py:648-653, 314-341) ------------------------------------
    // Roles by thread (the same for every track, one track at a time: values first, stores after):
    //   tid < 36      group dispersion entry (_estimate_group_disp_matrix 292-297)
    //   64 <= tid < 70  centroid, extrema, spread of dimension tid - 64 (_estimate_measurement_spread 246-268)
    //   tid == 96     ring bookkeeping, lifetime, point count, status, N_est (_estimate_point_num 232-244)
    int ring_rows = 0;
    for (int j = 0; j < T0; ++j) {
        TrackRec& t = tr[j];
        const int n = misc[kBaseG + (ntiles & 1) * 32 + j];
        ring_rows += n < kFeatPts ? n : kFeatPts;
        if (n == 0) {
            if (tid == 96) t.lifetime += dt;                     // update_lifetime(dt) (400-407)
            continue;
        }
        const double* tv = Bm + j * kBw;
        const double dn = (double)n;
        double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
        if (tid < 36) {
            double n_est;
            if (c.enable_est) n_est = dn > t.n_est ? dn : (1 - c.a_n) * t.n_est + c.a_n * dn;
            else n_est = (double)(n > c.est_pointnum ? n : c.est_pointnum);
            int r = el.i6, q = el.a6;
            if (r > q) { const int tmp = r; r = q; q = tmp; }
            const int p = r * 6 - (r * (r - 1)) / 2 + (q - r);
            const double rn = 1.0 / dn;
            const double dv = tv[kProd + p] * rn - (tv[kSum + r] * rn) * (tv[kSum + q] * rn);
            const double al = dn / n_est;
            v0 = (1 - al) * t.G[tid] + al * dv;
        } else if (tid >= 64 && tid < 70) {
            const int m = tid - 64;
            const double mnv = tv[kMin + m], mxv = tv[kMax + m];
            // centroid[0]: the x column is a sum of lattice values, exact in any order, so this is numpy's mean to the
            // bit -- the pose features sort on x - centroid[0] against zero pads (Utils.py:505-514)
            v0 = m == 0 ? tv[kSumX] / dn : tv[kHx + m] + tv[kSum + m] / dn;
            v1 = mnv;
            v2 = mxv;
            double spread = mxv - mnv;
            if (n != 1) spread = spread * (double)(n + 1) / (double)(n - 1);
            spread = fmin(2 * c.spread_lim[m], spread);
            spread = fmax(c.spread_lim[m], spread);
            v3 = spread > t.spread[m] ? spread : (1.0 - c.a_spr) * t.spread[m] + c.a_spr * spread;
        } else if (tid == 96) {
            if (c.enable_est) v0 = dn > t.n_est ? dn : (1 - c.a_n) * t.n_est + c.a_n * dn;
            else v0 = (double)(n > c.est_pointnum ? n : c.est_pointnum);
            const double c3 = tv[kHx + 3] + tv[kSum + 3] / dn, c4 = tv[kHx + 4] + tv[kSum + 4] / dn,
                         c5 = tv[kHx + 5] + tv[kSum + 5] / dn;
            v1 = sqrt(c3 * c3 + c4 * c4 + c5 * c5) < c.vel_thres ? 1.0 : 0.0;
        }
        if (tid < 36) {
            t.G[tid] = v0;
        } else if (tid >= 64 && tid < 70) {
            const int m = tid - 64;
            t.centroid[m] = v0; t.minv[m] = v1; t.maxv[m] = v2; t.spread[m] = v3;
        } else if (tid == 96) {
            const int phys = t.ring_n >= c.ring_size ? t.ring_head : ring_wrap(t.ring_head + t.ring_n, c.ring_size);
            if (t.ring_n >= c.ring_size) t.ring_head = ring_wrap(t.ring_head + 1, c.ring_size);
            else t.ring_n += 1;
            t.ring_cnt[phys] = n < kFeatPts ? n : kFeatPts;
            t.lifetime = 0.0;
            t.point_num = n;
            t.is_static = v1 != 0.0 ? 1 : 0;
            t.n_est = v0;         // (the dispersion threads computed their own copy from the old value above)
        }
    }
    {
        if (!sc.ring_ph_gone && sc.ring_n + 1 >= c.ring_size) sc.ring_ph_gone = 1;   // the deque's initial empty frame
        if (sc.ring_n >= c.ring_size) sc.ring_head = ring_wrap(sc.ring_head + 1, c.ring_size);
        else sc.ring_n += 1;
        sc.ring_cnt[uphys] = U;
    }
    // this frame's cell histogram takes the ring slot of the frame just pushed: saturating bytes, in shared memory
    // for the screen below and in global memory for the next two frames
    if (tid <= 64) {
        unsigned wd;
        if (tid < 64) {
            const unsigned lo = reinterpret_cast<const unsigned*>(hnew)[2 * tid], hi = reinterpret_cast<const unsigned*>(hnew)[2 * tid + 1];
            const unsigned c0 = min(lo & 0xffffu, 255u), c1 = min(lo >> 16, 255u), c2 = min(hi & 0xffffu, 255u),
                           c3 = min(hi >> 16, 255u);
            wd = c0 | (c1 << 8) | (c2 << 16) | (c3 << 24);
        } else {
            wd = misc[kFlag] ? 1u : 0u;
        }
        reinterpret_cast<unsigned*>(hist + uphys * kHistBytes)[tid] = wd;
        reinterpret_cast<unsigned*>(a.ring_hist + ((size_t)s * kRing + uphys) * kHistBytes)[tid] = wd;
    }
    __syncthreads();
    PHASE_MARK(8);

    // ---- 4. maintenance (Tracking.py:513-528, Q16): drop timed-out tracks, keep list order -------------------
    if (warp == 0) {
        bool kp = false;
        unsigned slotbit = 0u;
        if (lane < T0) {
            const double lim = tr[lane].is_static ? c.life_sta : c.life_dyn;
            kp = !(tr[lane].lifetime > lim);                     // dropped tracks are INACTIVE: off the list
            if (!kp) slotbit = 1u << tr[lane].slot;
        }
        const unsigned kmask = __ballot_sync(kFull, kp);
        const unsigned freed = __reduce_or_sync(kFull, slotbit);
        if (kp) misc[kOrder + __popc(kmask & ltmask)] = lane;
        if (lane == 0) { misc[kT1] = __popc(kmask); misc[kFreed] = (int)freed; }
    }
    __syncthreads();
    const int T1 = misc[kT1];
    sc.slot_mask &= ~(unsigned)misc[kFreed];
    PHASE_MARK(9);

    // ---- 5. update every surviving track (Tracking.py:598-603, 387-398; Q11-Q13) ----------------------------
    // Element-parallel steps of the Joseph-form update (linalg.cuh), one track at a time in each step.
    // _get_Rc (299-312): Rm/N + ((N_est - N)/((N_est - 1) N)) * group_disp_est;  S = P[:6,:6] + Rc
    for (int k = 0; k < T1; ++k) {
        if (tid < 36) {
            const int j = misc[kOrder + k];
            const TrackRec& t = tr[j];
            const double Nn = (double)t.point_num;
            const double coef = div_zero_fast(t.n_est - Nn, (t.n_est - 1.0) * Nn);     // N_est == N: zero numerator
            double rm = 0.0;
            if (el.i6 == el.a6) { const double h = t.spread[el.i6] / 2; rm = (h * h) / Nn; }
            const double rc = rm + coef * t.G[tid];
            double* b = Bm + j * kBw;
            b[36 + tid] = rc;
            b[tid] = t.P[el.i6 * 9 + el.a6] + rc;
        }
    }
    __syncthreads();
    for (int k0 = 0; k0 < T1; k0 += 2 * kStepWarps) {
        const int k = k0 + 2 * warp + (lane >> 4);
        const bool live = k < T1;
        if (__ballot_sync(kFull, live) == 0u) continue;
        const int j = live ? misc[kOrder + k] : 0;
        double r[6];
        (void)inv6_spd_half(live ? Bm + j * kBw : nullptr, lane, r);
        __syncwarp();
        const int cl16 = lane & 15;
        if (live && cl16 >= 6 && cl16 < 12) {
#pragma unroll
            for (int i = 0; i < 6; ++i) Bm[j * kBw + i * 6 + (cl16 - 6)] = r[i];
        }
    }
    __syncthreads();
    for (int k = 0; k < T1; ++k) {                       // K = P[:, :6] S^-1
        const int j = misc[kOrder + k];
        if (tid < 54) KKm[j * 108 + tid] = kf_update_K_elem(tr[j].P, Bm + j * kBw, el);
    }
    __syncthreads();
    for (int k = 0; k < T1; ++k) {                       // M1 = (I - K H) P, K Rc, x += K y
        const int j = misc[kOrder + k];
        TrackRec& t = tr[j];
        const double* K = KKm + j * 108;
        double mv = 0.0, rv = 0.0, xv = 0.0;
        if (tid < 81) mv = kf_update_M1_elem(t.P, K, el);
        if (tid < 54) rv = kf_update_KR_elem(K, Bm + j * kBw + 36, el);
        if (tid >= 96 && tid < 105) xv = kf_update_x(t.x, t.centroid, K, tid - 96);
        __syncwarp();                    // warp 3: every lane has read the old x
        if (tid < 81) Am[j * 81 + tid] = mv;
        if (tid < 54) KKm[j * 108 + 54 + tid] = rv;
        if (tid >= 96 && tid < 105) t.x[tid - 96] = xv;
    }
    __syncthreads();
    for (int k = 0; k < T1; ++k) {                       // P = M1 (I - K H)' + (K Rc) K'
        const int j = misc[kOrder + k];
        TrackRec& t = tr[j];
        if (tid < 81) t.P[tid] = kf_update_P_elem(Am + j * 81, KKm + j * 108, KKm + j * 108 + 54, el);
        if (tid == 96) kf_update_nudge(t.x, t.centroid, t.lifetime == 0.0, c.nudge_thres, c.nudge_gain);
    }
    PHASE_MARK(10);

    // ---- 6. DBSCAN over the fused global ring (Tracking.py:693-700): the grid screen --------------------------
    int Bf = 0;
    int fphys[kRing];
    bool fl = false;
    for (int f = 0; f < kRing; ++f) {
        fphys[f] = ring_wrap(sc.ring_head + f, c.ring_size);
        if (f < sc.ring_n) {
            Bf += sc.ring_cnt[fphys[f]];
            fl = fl || hist[fphys[f] * kHistBytes + kGridCells] != 0;
        }
    }
    const bool run_db = Bf > 0 && T1 < c.tr_max_tracks;
    if (run_db) {
        // The residue of a steady scene cannot hold a core point and is all noise (dbscan.cuh): 99.9 % of the
        // scene-frames.  Whatever the screen lets through is most likely a cluster forming -- a couple of scenes per
        // frame -- and goes to dbscan_big_kernel (512 threads per scene) through the work list.
        bool maybe = Bf >= c.db_min_samples;
        if (maybe && c.grid_ok && !fl) {
            // (the counts of this frame were packed before the barrier that followed the association results)
            for (int cell = tid; cell < kGridCells; cell += kStepThreads) {
                int n = 0;
                for (int f = 0; f < kRing; ++f)
                    if (f < sc.ring_n) n += hist[fphys[f] * kHistBytes + cell];
                hnew[cell] = (uint16_t)n;
            }
            __syncthreads();
            maybe = grid_screen_may_have_core(hnew, c.db_min_samples);
        }
        if (maybe) {
            if (tid == 0) a.defer_list[atomicAdd(a.defer_count, 1)] = s;
        } else if (a.labels_out != nullptr) {
            for (int b = tid; b < Bf; b += kStepThreads) a.labels_out[(size_t)s * 3 * ncap + b] = -1;
        }
        sc.dbscan_n = Bf;
    }
    __syncthreads();                     // the update's last step has written P
    PHASE_MARK(11);

    pdl_launch_dependents();             // late on purpose: dbscan_big's CTAs would otherwise sit on 16 SMs for the whole step
    // ---- 7. write back: track records in list order, scene record, per-scene counters --------------------------
    {
        double* dstbase = reinterpret_cast<double*>(a.tracks + (size_t)s * tcap);
        for (int i = tid; i < T1 * kTrackWords; i += kStepThreads) {
            const int k = i / kTrackWords, wd = i - k * kTrackWords;
            dstbase[i] = reinterpret_cast<const double*>(tr + misc[kOrder + k])[wd];
        }
    }
    if (tid == 0) {
        sc.n_tracks = T1;
        a.scenes[s] = sc;
        a.pose_cnt[s] = T1;
        int4* st4 = reinterpret_cast<int4*>(a.scene_stats + (size_t)s * 8);
        st4[0] = make_int4(N, M, U, run_db ? Bf : 0);
        st4[1] = make_int4(T1, ring_rows, 1, 0);
    }
    PHASE_MARK(12);
    if (dbg_clocks && threadIdx.x == 0) {
        a.phase_cycles[16 + blockIdx.x] = (unsigned long long)(clock64() - kernel_t0);   // last frame's cycles of this scene
        unsigned long long ns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
        a.phase_cycles[16 + 2 * gridDim.x + blockIdx.x] = ns;
    }
}

// DBSCAN + spawn for the scenes whose fused cloud passed the step kernel's grid screen (a cluster is forming: a
// couple of scenes per frame): one CTA of 512 threads per scene, new tracks written straight to the scene's list in
// global memory.  The last CTA also folds the step's per-scene counters into the context's totals.
constexpr int kBigThreads = 512;
constexpr int kBitsMaxB = 768;        // adjacency bit matrix of up to 768 x 768 (72 KB of shared memory)
__host__ __device__ inline int big_bits_cap(int ncap) { return 3 * ncap < kBitsMaxB ? 3 * ncap : kBitsMaxB; }
// shared-memory layout of dbscan_big_kernel: Xf|Yf|Zf, par, cl, scan, adj, cm, ws, raw rows, (8-byte aligned) w6
constexpr int kBigWsWords = 4 + kMaxCompMasks;    // per-word scratch rows of dbscan_bits_block
__host__ __device__ inline int big_adj_offset(int ncap) { return 36 * ncap + 2 * 3 * ncap * 4 + 64 * 4; }
__host__ __device__ inline int big_w6_offset(int ncap) {
    const int cap = big_bits_cap(ncap), w = (cap + 31) / 32;
    const int o = 36 * ncap + 2 * 3 * ncap * 4 + 64 * 4 + (cap * w + (1 + kBigWsWords) * w) * 4 + cap * kRawCols * 4;
    return (o + 7) & ~7;
}
__global__ void __launch_bounds__(kBigThreads, 1) dbscan_big_kernel(const __grid_constant__ StepArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    const DevConfig& c = a.cfg;
    const int ncap = c.ncap, tcap = c.tcap;
    float* Xf = reinterpret_cast<float*>(smem);
    int* par = reinterpret_cast<int*>(smem + 36 * ncap);
    int* cl = par + 3 * ncap;
    int* scan = cl + 3 * ncap;                               // 64 ints
    // bit-matrix DBSCAN (dbscan.cuh) for fused clouds of up to kBitsMaxB points; larger ones (dense configurations
    // with > 256 points per frame) take the pair-sweep version
    const int bits_cap = big_bits_cap(ncap), bits_w = (bits_cap + 31) >> 5;
    unsigned* adj = reinterpret_cast<unsigned*>(scan + 64);
    unsigned* cm = adj + (size_t)bits_cap * bits_w;
    unsigned* bws = cm + bits_w;                             // kBigWsWords rows of bits_w words
    float* rawc = reinterpret_cast<float*>(bws + kBigWsWords * bits_w);     // bits_cap raw rows
    double* w6 = reinterpret_cast<double*>(smem + big_w6_offset(ncap));   // bits_cap world 6-vectors
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    pdl_wait();                          // step_kernel has completed: work list, scene and track records are final
    pdl_launch_dependents();
    const int n_defer = *a.defer_count;
    // debug accounting (mmw_dbscan_big_clocks): cycles of thread 0 per part, summed over the deferred scenes
    unsigned long long* dbg = a.phase_cycles != nullptr ? a.phase_cycles + 16 + 3 * a.n_scenes : nullptr;
    long long dbg_t = clock64();
    auto stamp = [&](int k) {
        if (dbg != nullptr && tid == 0) {
            const long long now = clock64();
            atomicAdd(&dbg[k], (unsigned long long)(now - dbg_t));
            dbg_t = now;
        }
    };
    __shared__ SensorRec s_sr;            // the scene's mounting
    for (int it = blockIdx.x; it < n_defer; it += gridDim.x) {
        const int s = a.defer_list[it];
        SceneRec sc = a.scenes[s];
        if (tid < (int)(sizeof(SensorRec) / 8))
            reinterpret_cast<double*>(&s_sr)[tid] = reinterpret_cast<const double*>(a.sensors + s)[tid];
        __syncthreads();
        const int T1 = sc.n_tracks;
        int B = 0;
        int fcnt[kRing], fphys[kRing];
        for (int f = 0; f < kRing; ++f) {
            fphys[f] = ring_wrap(sc.ring_head + f, c.ring_size);
            fcnt[f] = f < sc.ring_n ? sc.ring_cnt[fphys[f]] : 0;
            B += fcnt[f];
        }
        const bool bits = B <= bits_cap;
        NbScreened nb = load_fused_ring(a, s_sr, s, fcnt, fphys, Xf, 3 * ncap, bits ? rawc : nullptr);
        stamp(0);
        int ncl = bits ? dbscan_bits_block(nb, B, c.db_min_samples, adj, cm, bws, par, cl, dbg != nullptr ? dbg - 10 : nullptr)
                       : dbscan_block(nb, B, c.db_min_samples, par, cl, scan, dbg != nullptr ? dbg - 10 : nullptr, false,
                                      true);
        if (dbg != nullptr && tid == 0) dbg_t = clock64();
        if (a.labels_out != nullptr)
            for (int b = tid; b < B; b += kBigThreads) a.labels_out[(size_t)s * 3 * ncap + b] = cl[b];
        if (ncl > 0) {
            if (T1 + ncl > tcap) { ncl = tcap - T1; sc.flags |= MMW_SCENE_TRACK_OVERFLOW; }
            int newslot[kMaxTcap];
            {
                const unsigned capmask = tcap >= 32 ? 0xffffffffu : ((1u << tcap) - 1u);
                unsigned fs = ~sc.slot_mask & capmask;
                for (int q = 0; q < ncl; ++q) {
                    newslot[q] = __ffs(fs) - 1; fs &= fs - 1;
                    sc.slot_mask |= 1u << newslot[q];
                }
            }
            if (bits) {                  // world coordinates and velocities of the clustered points, all threads
                for (int b = tid; b < B; b += kBigThreads)
                    if (cl[b] >= 0) {
                        const float* r = rawc + (size_t)b * kRawCols;
                        double w[6];
                        world_from_raw(s_sr, r[0], r[1], r[2], r[3], w);
#pragma unroll
                        for (int k = 0; k < 6; ++k) w6[(size_t)b * 6 + k] = w[k];
                    }
                __syncthreads();
            }
            if (bits) {
                // the adjacency matrix is dead by now: its first bytes serve as the reduction scratch
                double* red = reinterpret_cast<double*>(adj);
                for (int q = 0; q < ncl; ++q)
                    spawn_track_block(a, s, a.tracks[(size_t)s * tcap + T1 + q], q, newslot[q], sc.next_id + q, cl, B, rawc,
                                      w6, red);
            } else {
                for (int q = warp; q < ncl; q += kBigThreads / 32)
                    spawn_track(a, s_sr, s, a.tracks[(size_t)s * tcap + T1 + q], q, newslot[q], sc.next_id + q, cl, fcnt,
                                fphys, lane, nullptr, nullptr);
            }
            if (a.nr_extra != nullptr) {
                // Pose rows of the new tracks, behind the rows of all tracks that existed when step_kernel finished (the
                // feature kernel lays those out, concurrently): R0 = sum of pose_cnt, which this kernel leaves alone
                __shared__ int s_part[kBigThreads / 32], s_row0;
                __syncthreads();                                     // the spawns' global writes are visible to the CTA
                int part = 0;
                for (int i = tid; i < a.n_scenes; i += kBigThreads) part += a.pose_cnt[i];
                part = __reduce_add_sync(kFullMask, part);
                if (lane == 0) s_part[warp] = part;
                __syncthreads();
                if (tid == 0) {
                    int r0 = 0;
                    for (int w = 0; w < kBigThreads / 32; ++w) r0 += s_part[w];
                    s_row0 = r0 + atomicAdd(a.nr_extra, ncl);
                }
                __syncthreads();
                const int nfr = c.ring_size;
                unsigned char* scratch = smem + ((big_adj_offset(ncap) + 15) & ~15) + warp * kFeatItemBytes;
                long long* fkeys = reinterpret_cast<long long*>(scratch);
                float* fso = reinterpret_cast<float*>(scratch + kFeatPts * 8);
                uint4* fsp = reinterpret_cast<uint4*>(scratch + kFeatPts * 8 + kFeatPts * kRawCols * 4);
                for (int item = warp; item < ncl * nfr; item += kBigThreads / 32) {
                    const int q = item / nfr, f = item - q * nfr, row = s_row0 + q, slot = newslot[q];
                    const TrackRec* t = a.tracks + (size_t)s * tcap + T1 + q;
                    if (f == 0 && lane == 0) {
                        a.nr_row_scene[row] = s; a.nr_row_track[row] = T1 + q; a.nr_row_slot[row] = slot;
                    }
                    // a fresh track's ring holds one frame: the first 64 cluster rows (spawn_track*); the others are zero
                    const float* src = f == 0 ? a.track_ring + ((size_t)s * tcap + slot) * kRing * (kFeatPts * kRawCols) : nullptr;
                    const int cnt = f == 0 ? __ldcg(&t->ring_cnt[0]) : 0;
                    float* out = a.nr_feats + ((size_t)row * nfr + f) * (kFeatPts * kRawCols);
                    uint4* pk = a.nr_packed != nullptr
                                    ? reinterpret_cast<uint4*>(static_cast<unsigned char*>(a.nr_packed) + (size_t)row * nfr * kFeatPts * 32)
                                    : nullptr;
                    pose_feature_item<false>(c, s_sr, src, cnt, __ldcg(&t->centroid[0]), __ldcg(&t->centroid[1]), f, out, pk,
                                             fkeys, fso, fsp, lane, 0);
                }
            }
            sc.next_id += ncl;
            sc.n_tracks = T1 + ncl;
            sc.ring_n = 0;               // batch.clear() (Tracking.py:699-700, Q8)
            sc.ring_head = 0;
            sc.ring_cnt[0] = sc.ring_cnt[1] = sc.ring_cnt[2] = 0;
            sc.ring_ph_gone = 1;
            if (tid == 0) atomicAdd(&a.counters[5], (unsigned long long)ncl);
        }
        __syncthreads();
        if (tid == 0) { a.scenes[s] = sc; if (a.nr_extra == nullptr) a.pose_cnt[s] = sc.n_tracks; }
        __syncthreads();
        stamp(1);
        if (dbg != nullptr && tid == 0) { atomicAdd(&dbg[2], 1ull); atomicAdd(&dbg[7], (unsigned long long)B); }
    }
    // this step's counters: every scene left eight ints; the grid's last CTA (idle unless 16 clusters form at once)
    // sums them -- one reduction and seven atomics per step instead of seven atomics per scene
    if (blockIdx.x == gridDim.x - 1 && a.scene_stats != nullptr) {
        unsigned long long acc[7] = {0, 0, 0, 0, 0, 0, 0};
        for (int sidx = tid; sidx < a.n_scenes; sidx += kBigThreads) {
            const int4 s0 = reinterpret_cast<const int4*>(a.scene_stats)[2 * sidx];
            const int4 s1 = reinterpret_cast<const int4*>(a.scene_stats)[2 * sidx + 1];
            acc[0] += (unsigned)s1.z; acc[1] += (unsigned)s0.x; acc[2] += (unsigned)s0.y; acc[3] += (unsigned)s0.z;
            acc[4] += (unsigned)s0.w; acc[5] += (unsigned)s1.x; acc[6] += (unsigned)s1.y;
        }
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            unsigned v = (unsigned)acc[k];                   // < 2^32 per thread: at most S / 512 scenes of < 2^16 each
            v = __reduce_add_sync(kFullMask, v);
            if (lane == 0 && v) atomicAdd(&a.counters[k], (unsigned long long)v);
        }
    }
    // every CTA read the work-list length when it started; the last one to finish empties the list for the next step
    // (no memset node between the steps)
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(a.defer_done, 1) == (int)gridDim.x - 1) {
            if (a.defer_hint != nullptr) *a.defer_hint = n_defer;     // zero-copy write to pinned host memory
            *a.defer_count = 0;
            *a.defer_done = 0;
        }
    }
}

// after DBSCAN and the spawns, everything from the adjacency matrix on is scratch for the new tracks' feature maps
// (one kFeatItemBytes block per warp)
int dbscan_big_smem_bytes(int ncap) {
    const int a = big_w6_offset(ncap) + big_bits_cap(ncap) * 6 * 8;
    const int b = ((big_adj_offset(ncap) + 15) & ~15) + (kBigThreads / 32) * kFeatItemBytes;
    return a > b ? a : b;
}

cudaError_t launch_step(const StepArgs& a, cudaStream_t stream) {
    const int smem = step_smem_bytes(a.cfg.ncap, a.cfg.tcap);
    static int configured[kMaxDevices] = {0};
    cudaError_t e = ensure_smem_attr(reinterpret_cast<const void*>(step_kernel), configured, smem);
    if (e != cudaSuccess) return e;
    step_kernel<<<a.n_scenes, kStepThreads, smem, stream>>>(a);
    return cudaGetLastError();
}

// grid: 16 CTAs cover the couple of scenes per frame in which a cluster forms (C2); dense configurations keep every
// scene's DBSCAN busy (untracked targets stay in the residue) and get one CTA per SM -- chosen by the caller from the
// work-list length of an earlier step (StepArgs::defer_hint), which only affects speed, never results.
cudaError_t launch_dbscan_big(const StepArgs& a, cudaStream_t stream, int grid) {
    if (a.defer_count == nullptr) return cudaSuccess;
    const int big_smem = dbscan_big_smem_bytes(a.cfg.ncap);
    static int configured[kMaxDevices] = {0};
    cudaError_t e = ensure_smem_attr(reinterpret_cast<const void*>(dbscan_big_kernel), configured, big_smem);
    if (e != cudaSuccess) return e;
    return launch_pdl(dbscan_big_kernel, dim3(grid < 16 ? 16 : (grid > 148 ? 148 : grid)), dim3(kBigThreads), big_smem, stream,
                      dim3(1, 1, 1), a);
}

}  // namespace mmw
