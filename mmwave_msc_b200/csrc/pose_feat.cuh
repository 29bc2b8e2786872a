// pose_feature_item: relative_coordinates + format_single_frame (Utils.py:437-520) for one ring frame of one track, by
// one warp.  Used by pose_feature_kernel (pose_kernels.cu) and by dbscan_big_kernel (step_kernel.cu) for the tracks it
// has just spawned.
#pragma once
#include <cuda_bf16.h>

#include "mmw_internal.cuh"

namespace mmw {

// The feature maps of ONE ring frame of one track by one warp (shared by pose_feature_kernel and, for the tracks it
// has just spawned, dbscan_big_kernel): sr = the scene's mounting and Doppler unit, src = the frame's 64 raw rows in
// the track's ring (nullptr: the frame is not in the ring yet, its maps are zero), cnt real rows, (cx, cy) the track's
// CURRENT centroid.  Scratch per warp: 64 int64 keys, 320 floats, 128 uint4 (kFeatItemBytes).  kReadOnly: the rows
// were written by an earlier kernel (ld.global.nc).
constexpr int kFeatItemBytes = kFeatPts * 8 + kFeatPts * kRawCols * 4 + kFeatPts * 2 * 16;
template <bool kReadOnly>
__device__ __forceinline__ void pose_feature_item(const DevConfig& c, const SensorRec& sr, const float* src, int cnt,
                                                  double cx, double cy, int f, float* out, uint4* pk, long long* keys,
                                                  float* so, uint4* spk_w, int lane, int dbg) {
    if (src == nullptr) {
        for (int e = lane; e < kFeatPts * kRawCols; e += 32) out[e] = 0.f;
        if (pk)
            for (int e = lane; e < kFeatPts * 2; e += 32) pk[f * kFeatPts * 2 + e] = make_uint4(0, 0, 0, 0);
        return;
    }
    {   // the frame's 64 raw rows (1280 contiguous bytes) as 80 float4 loads, not 10 strided scalar loads per lane
        const float4* g4 = reinterpret_cast<const float4*>(src);
        float4* s4 = reinterpret_cast<float4*>(so);
        if (!(dbg & 8))
            for (int e = lane; e < kFeatPts * kRawCols / 4; e += 32) s4[e] = kReadOnly ? __ldg(g4 + e) : __ldcg(g4 + e);
    }
    __syncwarp();
    float v[2][kRawCols];
    long long mkey[2];
    // Fast path of the sort (taken when every x of the frame is a multiple of 2^-16 below 128 m -- the sensor's
    // Q-format lattice -- and |cx| < 2^30): there fl(x - cx) is STRICTLY monotone in x (two lattice values differ by
    // >= 2^-16, the rounding moves a difference by < 2^-22), and a pad (key 0.0) sorts like a point at cx.  So the
    // order of (key, index) is the order of the 32-bit word  (2 x 2^16 [pads: the odd or even integer at cx] + 2^25)
    // << 6 | index, all different: one integer compare per pair instead of a 64-bit compare with a tie rule.
    int kx[2];
    bool lattice = fabs(cx) < 1073741824.0;
    {
        const double cs = cx * 65536.0, fl = floor(cs);
        const int kpad = cs >= 8388608.0 ? (1 << 24) + 1 : (cs <= -8388608.0 ? -(1 << 24) - 1
                         : 2 * (int)fl + (cs != fl ? 1 : 0));
        kx[0] = kx[1] = kpad;
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int i = lane + 32 * h;
        double key = 0.0;
#pragma unroll
        for (int q = 0; q < kRawCols; ++q) v[h][q] = 0.f;
        if (i < cnt) {
            {
                const float xs = so[i * kRawCols + 0] * 65536.f;
                lattice = lattice && fabsf(xs) < 8388608.f && xs == rintf(xs);
                kx[h] = 2 * (int)xs;
            }
            const float x = so[i * kRawCols + 0], y = so[i * kRawCols + 1], z = so[i * kRawCols + 2];
            const float d = so[i * kRawCols + 3], p = so[i * kRawCols + 4];
            double yw, zw;
            const SensorRec m = sensor_at_use(sr);
            world_yz(m, (double)y, (double)z, yw, zw);
            key = __dsub_rn((double)x, cx);
            v[h][0] = (float)key;
            v[h][1] = (float)__dsub_rn(yw, cy);
            v[h][2] = (float)zw;
            v[h][3] = (float)__dmul_rn((double)d, m.doppler_res);
            v[h][4] = (float)__ddiv_rn(__dsub_rn((double)p, c.int_mu), c.int_std);
        }
        const long long b = __double_as_longlong(__dadd_rn(key, 0.0));
        mkey[h] = b ^ ((b >> 63) & 0x7fffffffffffffffLL);
    }
    const bool fast = __all_sync(0xffffffffu, lattice) && !(dbg & 16);
    if (!fast) {
        keys[lane] = mkey[0];
        keys[lane + 32] = mkey[1];
    } else {
        unsigned* k32 = reinterpret_cast<unsigned*>(keys);
        k32[lane] = ((unsigned)(kx[0] + (1 << 25)) << 6) | (unsigned)lane;
        k32[lane + 32] = ((unsigned)(kx[1] + (1 << 25)) << 6) | (unsigned)(lane + 32);
    }
    __syncwarp();
    int rank[2] = {0, 0};
    if (fast) {
        const unsigned c0 = ((unsigned)(kx[0] + (1 << 25)) << 6) | (unsigned)lane;
        const unsigned c1 = ((unsigned)(kx[1] + (1 << 25)) << 6) | (unsigned)(lane + 32);
        const uint4* k4 = reinterpret_cast<const uint4*>(keys);
#pragma unroll
        for (int q4 = 0; q4 < kFeatPts / 4; ++q4) {
            const uint4 kq = k4[q4];                 // broadcast read
            rank[0] += (kq.x < c0) + (kq.y < c0) + (kq.z < c0) + (kq.w < c0);
            rank[1] += (kq.x < c1) + (kq.y < c1) + (kq.z < c1) + (kq.w < c1);
        }
    } else {
    // Stable rank of (key, index).  Float64 compares (DSETP) issue at a fraction of the integer rate on this part
    // and the 4096 compares per frame were two thirds of the kernel's time (profiles/r02_feat_probe.txt), so the
    // keys are compared as integers: a finite double maps to an int64 with the same order (-0.0 was folded into
    // +0.0 above), and "kq < k  or  (kq == k and q < i)" is "mq < m + (q < i)".
    const long long lt0 = mkey[0], le0 = mkey[0] + 1, lt1 = mkey[1], le1 = mkey[1] + 1;
    const longlong2* k2 = reinterpret_cast<const longlong2*>(keys);
    const int nq2 = (dbg & 4) ? 1 : kFeatPts / 4;
#pragma unroll 8
    for (int q2 = 0; q2 < nq2; ++q2) {               // q = 2 q2, 2 q2 + 1 < 32: below every index of the second point
        const longlong2 kq = k2[q2];                 // broadcast read
        const int q = 2 * q2;
        rank[0] += kq.x < (q < lane ? le0 : lt0) ? 1 : 0;
        rank[0] += kq.y < (q + 1 < lane ? le0 : lt0) ? 1 : 0;
        rank[1] += kq.x < le1 ? 1 : 0;
        rank[1] += kq.y < le1 ? 1 : 0;
    }
#pragma unroll 8
    for (int q2 = 0; q2 < nq2; ++q2) {               // q = 32 + 2 q2 ...: above every index of the first point
        const longlong2 kq = k2[kFeatPts / 4 + q2];
        const int q = 2 * q2;
        rank[0] += kq.x < lt0 ? 1 : 0;
        rank[0] += kq.y < lt0 ? 1 : 0;
        rank[1] += kq.x < (q < lane ? le1 : lt1) ? 1 : 0;
        rank[1] += kq.y < (q + 1 < lane ? le1 : lt1) ? 1 : 0;
    }
    }
    // the sorted frame is put together in shared memory and leaves as whole 16-byte vectors: a row is 20 bytes,
    // written from registers it cost 14 store instructions of 32 scattered sectors each (the L2 request rate, not
    // the bytes, bounded the kernel)
    uint4* sp = spk_w;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int q = 0; q < kRawCols; ++q) so[rank[h] * kRawCols + q] = v[h][q];
        if (pk) {
            __align__(16) __nv_bfloat16 pv[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) pv[q] = __float2bfloat16_rn(0.f);
#pragma unroll
            for (int q = 0; q < kRawCols; ++q) {
                const float x = v[h][q];
                pv[q] = __float2bfloat16_rn(x);
                pv[8 + q] = __float2bfloat16_rn(x - __bfloat162float(pv[q]));
            }
            // slab order of the tensor-core convs: [row][d = f][w][chunk][h][8]  (pose_tc.cu)
            const int ph = rank[h] >> 3, pw_ = rank[h] & 7;
            sp[(pw_ * 2 + 0) * 8 + ph] = reinterpret_cast<const uint4*>(pv)[0];
            sp[(pw_ * 2 + 1) * 8 + ph] = reinterpret_cast<const uint4*>(pv)[1];
        }
    }
    __syncwarp();
    if (!(dbg & 2)) {
        float4* o4 = reinterpret_cast<float4*>(out);
        const float4* s4 = reinterpret_cast<const float4*>(so);
        for (int e = lane; e < kFeatPts * kRawCols / 4; e += 32) o4[e] = s4[e];
        if (pk) {
#pragma unroll
            for (int e = 0; e < 4; ++e) pk[f * kFeatPts * 2 + e * 32 + lane] = sp[e * 32 + lane];
        }
    }
    __syncwarp();                    // the keys are reused by this warp's next item
}

}  // namespace mmw
