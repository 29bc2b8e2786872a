// The pose network (train.py:33-106) on the 5th-generation tensor cores: tcgen05.mma + TMEM + TMA.
//
// Precision.  The network is fp32 in the reference (Keras default) and the joints must hold 1 mm.  A single bf16
// or tf32 pass does not (SURVEY.md section 7: 14 mm / 2 mm worst case), so every fp32 operand is split into two
// bf16 terms, a = a_hi + a_lo, w = w_hi + w_lo, and three products are accumulated in fp32 in TMEM:
//     a_hi*w_hi + a_lo*w_hi + a_hi*w_lo            (the dropped a_lo*w_lo term is ~2^-16 relative)
//
// Convolutions (conv_slab_kernel): shifted-window implicit GEMM -- every tap is a tcgen05.mma on a shifted
// shared-memory descriptor of a slab staged once per sample and kh (details at the kernel).  Per tap the B operand is
// the K' x N' matrix [[W_hi | W_lo], [W_hi | 0]], so one MMA chain produces a*W_hi in columns [0,C) and a_hi*W_lo in
// columns [C,2C); the epilogue adds the two halves, bias, ReLU (+ BatchNorm after conv2) and writes the next layer's
// split operand directly.
//
// Dense layers: dense 1 on 256 x BN tiles of CTA pairs (gemm_tc_pair_kernel, tcgen05.mma.cta_group::2), dense 2 on
// 128 x 64 tiles (gemm_tc_kernel), K blocks of 64 (SWIZZLE_128B); each pipeline stage holds the four operand tiles
// {A_hi, A_lo, W_hi, W_lo} of one K block (loaded once by TMA, used by three MMAs per 16-wide K step).
//
// Warp roles in the dense kernels: warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), warps 2-5 = epilogue.
// All kernels are links of the step's programmatic-dependent-launch chain (mmw_internal.cuh).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "pose_tc.cuh"

namespace mmw {

// ---- PTX wrappers ------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
            "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <uint32_t COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(COLS) : "memory");
}

// K-major operand tile in shared memory whose rows are exactly one swizzle span wide (SW bytes = 32, 64 or 128),
// written by TMA with the matching swizzle: 8-row atoms are 8*SW bytes apart (SBO); LBO unused; version 1 (sm_100).
template <int SW>
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    constexpr uint64_t layout = SW == 128 ? 2 : (SW == 64 ? 4 : 6);
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)(((8 * SW) >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;
    d |= layout << 61;
    return d;
}
// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, M = 128.
__device__ __forceinline__ constexpr uint32_t make_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

__device__ __forceinline__ void split2(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

// =====================================================================================================
// Convolution as a shifted-window implicit GEMM
// =====================================================================================================
// First version (git history, profiles/r01_ncu_full_tma_im2col_conv.md): one TMA box per tap and slice (im2col by
// tensor-map coordinates, zero padding by out-of-bounds fill).  Correct, but the TMA unit is row-rate bound on
// 32/64-byte rows (~5 cycles per row, 27x re-read): 193 us + 200 us for conv1 + conv2 at ~1900 rows.
//
// Current version: per sample the activation slab is staged ONCE per kh in {-1,0,+1} into shared memory by four
// producer warps (cp.async, 16 B each), zero-padded in d and w, in the un-swizzled UMMA core-matrix layout with
// h as the row inside an 8-row atom:
//        slab_kh[d' = 0..D+1][w'' = 0..9][chunk][h = 0..7][8 ch]     entry = act[d'-1][h + kh][w''-1]
// With output rows ordered (d, w'', h) every tap (kd, kh, kw) is the SAME tile shifted by (1+kd)*10 + kw whole
// atoms inside slab_kh -- so all 27 taps are tcgen05.mma instructions on shifted shared-memory descriptors, and
// nobody copies im2col columns.  Output columns w'' = 0 and 9 are padding (discarded), i.e. 240 of the 256 MMA
// rows per sample are computed and 192 kept.  The three kh slabs form a ring: slab_kh of the next sample is
// refilled while the other two are still being multiplied.
struct ConvTcArgs {
    const int* n_rows;
    const float *bias, *bn_scale, *bn_shift;       // bn_* only for MODE 1
    const __nv_bfloat16* in;                       // packed input  [row][D][8][8][CK]  (hi | lo per position)
    __nv_bfloat16* out0;                           // MODE 0: act1 packed [row][D][8][8][32]; MODE 1: A_hi [row][Kf]
    __nv_bfloat16* out1;                           // MODE 1: A_lo [row][Kf]
    int dbg;                                       // timing experiments only (MMW_GEMM_DBG): 8 = producers idle,
                                                   // 16 = no MMAs, 32 = no epilogue stores
};

constexpr int kSlabThreads = 320;                  // warps 0-3 producers, 4-5 MMA issuers, 6-9 epilogue
constexpr int kSlabAtoms = 1 + 5 * 10 + 3;         // one guard atom in front, three behind (junk rows stay inside)

// Slab ring depth: the (sample, kh) uses form one sequence u = 3*n + c that cycles through NSLAB buffers, so the
// producers run up to NSLAB-1 uses ahead of the tensor core.
template <int CK>
__host__ __device__ constexpr int slab_ring() { return CK == 16 ? 8 : 4; }

// Weights of one tap in shared memory.  Conv 1 (CK = 16: ONE K16 MMA per tap holds a_hi and a_lo): [N = 2 cout][K16] with
// the (w_lo, a_lo) block zero.  Conv 2 (CK = 32: a K16 MMA for a_hi and one for a_lo): the a_hi MMA multiplies by
// [w_hi ; w_lo] (N = 64), the a_lo MMA only by w_hi (N = 32, accumulating into the first 32 columns) -- no zero block, 3 KB
// instead of 4 KB per tap and 5 KB instead of 6 KB of operand reads for every second MMA.
template <int CK, int NOUT>
__host__ __device__ constexpr int conv_b_tap_bytes() { return CK == 32 ? (NOUT + NOUT / 2) * 32 : NOUT * CK * 2; }
template <int CK, int NOUT>
constexpr int conv_smem_bytes_tc(int taps) {
    return taps * conv_b_tap_bytes<CK, NOUT>() + slab_ring<CK>() * kSlabAtoms * (CK / 8) * 128 + 1024 + 1024;
}

__device__ __forceinline__ uint64_t make_desc_interleaved(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;     // K direction: distance between 8x16B core matrices
    d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;     // M direction: distance between 8-row groups
    d |= (uint64_t)1 << 46;                         // version (sm_100); layout type 0 = no swizzle
    return d;
}

// Activations in HBM are stored in the slab's own order, [row][d][w][chunk][h][8 ch] (16-byte chunk = 8 bf16 of
// the hi|lo channel vector of one position), so the producers' global reads are fully coalesced and their
// shared-memory stores are bank-conflict free (8 consecutive lanes = the 128 contiguous bytes of one core matrix).
//
// CK   = K' per tap = 2 * padded input channels (hi | lo): 16 for conv1, 32 for conv2
// NOUT = MMA N     = 2 * output channels: 32 for conv1, 64 for conv2
// KD   = taps in depth.  A slab always holds D = 3 depth planes.  KD == 3: define_CNN_3D, one sample per slab.
// KD == 1: define_CNN, THREE consecutive samples ride as the three depth planes of one slab -- their packed inputs and
// outputs are contiguous in exactly the 3-D layout, the depth taps are simply not issued (9 taps, the d padding planes
// stay unused) -- 240 of 256 MMA rows used and a third of the per-sample hand-overs of one 8 x 8 map per slab: the C4
// configuration's convolutions went from 0.83 ms to the figure in DESIGN.md.  Samples past the row count in the last
// triple are staged as zeros and not stored.
template <int CK, int NOUT, int MODE, int KD>
__global__ void __launch_bounds__(kSlabThreads, 1)
conv_slab_kernel(const __grid_constant__ CUtensorMap map_b, const ConvTcArgs a) {
    constexpr int D = 3;                             // depth planes of a slab
    constexpr bool TRIPLE = KD == 1;
    constexpr int NCH = CK / 8;                      // 16-byte chunks per position
    constexpr int ATOM = NCH * 128;                  // bytes of one 8-row atom
    constexpr int SLAB_BYTES = kSlabAtoms * ATOM;
    constexpr int NSLAB = slab_ring<CK>();
    constexpr int B_TAP = conv_b_tap_bytes<CK, NOUT>();
    constexpr int B_ROWS = CK == 32 ? NOUT + NOUT / 2 : NOUT;        // rows of the weight tensor per tap
    constexpr int COUT = NOUT / 2;
    constexpr uint32_t TCOLS = 4 * NOUT;             // 2 accumulator buffers x 2 M tiles
    constexpr int taps = KD == 3 ? 27 : 9;
    constexpr int MT = 2;                            // M tiles of 128 rows per sample (or triple of samples)

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    unsigned char* sB = smem;
    unsigned char* slab = smem + taps * B_TAP;
    uint64_t* sfull = reinterpret_cast<uint64_t*>(slab + NSLAB * SLAB_BYTES);
    uint64_t* sempty = sfull + NSLAB;
    uint64_t* tfull = sempty + NSLAB;
    uint64_t* tempty = tfull + 2;
    uint64_t* bfull = tempty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + 1);
    float* sconst = reinterpret_cast<float*>(tmem_slot + 2);      // bias | bn_scale | bn_shift, COUT each

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // static zero padding (d, w borders and the h rows a shifted copy never receives)
    for (int i = threadIdx.x; i < NSLAB * SLAB_BYTES / 16; i += kSlabThreads)
        reinterpret_cast<uint4*>(slab)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x < COUT) {
        sconst[threadIdx.x] = a.bias[threadIdx.x];
        sconst[COUT + threadIdx.x] = MODE == 1 ? a.bn_scale[threadIdx.x] : 1.f;
        sconst[2 * COUT + threadIdx.x] = MODE == 1 ? a.bn_shift[threadIdx.x] : 0.f;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 4 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        for (int c = 0; c < NSLAB; ++c) { mbar_init(&sfull[c], 128); mbar_init(&sempty[c], MT); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], MT); mbar_init(&tempty[b], 4); }
        mbar_init(bfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // the layer's weights do not depend on the previous kernel: fetch them before the PDL wait below
        mbar_expect_tx(bfull, taps * B_TAP);
        for (int t = 0; t < taps; ++t) tma_load_2d(sB + t * B_TAP, &map_b, bfull, 0, t * B_ROWS);
    }
    if (warp == 4) tmem_alloc<TCOLS>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // everything above overlapped the previous kernel's tail (PDL); its activations and the row count are read below
    pdl_wait();
    pdl_launch_dependents();
    const int n_samples = *a.n_rows;
    const int rows = TRIPLE ? (n_samples + 2) / 3 : n_samples;        // slabs to process

    if (warp < 4) {
        // ===== producers: global -> registers (one sample ahead) -> the three h-shifted slabs of the sample =====
        constexpr int ITEMS = D * 64 * NCH / 128;            // 16-byte chunks per thread per sample
        const int tid = threadIdx.x;
        int dstoff[ITEMS];
        const int hsrc = tid & 7;                            // 128 % 8 == 0: every item of a thread has the same h
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
            const int i = tid + 128 * j;
            const int chunk = (i >> 3) % NCH, w = (i / (8 * NCH)) & 7, d = i / (64 * NCH);
            dstoff[j] = (1 + (d + 1) * 10 + (w + 1)) * ATOM + chunk * 128;
        }
        uint4 cur[ITEMS], nxt[ITEMS];
        auto load_row = [&](int row, uint4 (&r)[ITEMS]) {
            const uint4* src = reinterpret_cast<const uint4*>(a.in) + (size_t)row * (D * 64 * NCH);
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const bool there = !TRIPLE || row * 3 + (tid + 128 * j) / (64 * NCH) < n_samples;
                r[j] = there ? __ldg(src + tid + 128 * j) : make_uint4(0, 0, 0, 0);
            }
        };
        if ((int)blockIdx.x < rows && !(a.dbg & 8)) load_row(blockIdx.x, cur);
        int u = 0;
        for (int row = blockIdx.x; row < rows; row += gridDim.x) {
            const int next = row + gridDim.x;
            if (next < rows && !(a.dbg & 8)) load_row(next, nxt);
#pragma unroll
            for (int c = 0; c < 3; ++c, ++u) {
                const int slot = u % NSLAB;
                mbar_wait(&sempty[slot], (uint32_t)(((u / NSLAB) & 1) ^ 1));
                unsigned char* sl = slab + slot * SLAB_BYTES;
                const int hh = hsrc - (c - 1);               // this slab serves kh = c - 1: row h feeds output h - kh
                if (hh >= 0 && hh <= 7 && !(a.dbg & 8)) {
#pragma unroll
                    for (int j = 0; j < ITEMS; ++j) *reinterpret_cast<uint4*>(sl + dstoff[j] + hh * 16) = cur[j];
                }
                // the h row this copy never receives must be zero: it may hold the previous use's data
                const int hz = c == 0 ? 0 : (c == 2 ? 7 : -1);
                if (hz >= 0 && hsrc == hz) {
#pragma unroll
                    for (int j = 0; j < ITEMS; ++j)
                        *reinterpret_cast<uint4*>(sl + dstoff[j] + hz * 16) = make_uint4(0, 0, 0, 0);
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_arrive(&sfull[slot]);
            }
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) cur[j] = nxt[j];
        }
    } else if (warp == 4 || warp == 5) {
        // ===== MMA issuers: warp 4 owns M tile 0, warp 5 owns M tile 1 =====
        // Every operand address is slab/weight base + a compile-time constant, so one MMA costs two 64-bit adds.
        const int mt = warp - 4;
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(NOUT);
            constexpr uint32_t idesc_lo = make_idesc(NOUT / 2);                    // conv 2, a_lo chunk: N = cout
            const uint64_t db0 = make_desc<32>(smem_u32(sB));                      // weight rows are one K16 wide
            const uint64_t da00 = make_desc_interleaved(smem_u32(slab) + (uint32_t)((1 + mt * 16) * ATOM), 128, ATOM);
            mbar_wait(bfull, 0);
            int n = 0, u = 0;
            for (int row = blockIdx.x; row < rows; row += gridDim.x, ++n) {
                const int buf = n & 1;
                mbar_wait(&tempty[buf], (uint32_t)(((n >> 1) & 1) ^ 1));
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)((buf * 2 + mt) * NOUT);
#pragma unroll
                for (int c = 0; c < 3; ++c, ++u) {
                    const int slot = u % NSLAB;
                    mbar_wait(&sfull[slot], (uint32_t)((u / NSLAB) & 1));
                    tc_fence_after();
                    const uint64_t da0 = da00 + (uint64_t)((slot * SLAB_BYTES) >> 4);
#pragma unroll
                    for (int kdi = 0; kdi < (KD == 3 ? 3 : 1); ++kdi) {
#pragma unroll
                        for (int kwi = 0; kwi < 3; ++kwi) {
                            const int kd = KD == 3 ? kdi - 1 : 0, kw = kwi - 1;
                            const int tap = KD == 3 ? (kdi * 3 + c) * 3 + kwi : c * 3 + kwi;
                            const bool first = c == 0 && kdi == 0 && kwi == 0;
                            const int aoff = ((1 + kd) * 10 + kw) * ATOM;        // whole atoms: tap = tile shift
#pragma unroll
                            for (int kk = 0; kk < CK / 16; ++kk)
                                if (!(a.dbg & 16)) umma_bf16(tmem_d, da0 + (uint64_t)((aoff + kk * 256) >> 4),
                                          db0 + (uint64_t)((tap * B_TAP + kk * NOUT * 32) >> 4), kk == 0 ? idesc : idesc_lo,
                                          (first && kk == 0) ? 0u : 1u);
                        }
                    }
                    umma_commit(&sempty[slot]);   // the slab may be refilled once both issuers are done with it
                }
                umma_commit(&tfull[buf]);
            }
        }
    } else {
        // ===== epilogue: warps 6-9, TMEM lane quadrant = warp % 4 =====
        const int q = warp & 3;
        int n = 0;
        for (int row = blockIdx.x; row < rows; row += gridDim.x, ++n) {
            const int buf = n & 1;
            mbar_wait(&tfull[buf], (uint32_t)((n >> 1) & 1));
            tc_fence_after();
            float y[2][COUT];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * 2 + mt) * NOUT);
                uint32_t v[32];
                tmem_ld32(taddr, v);
                if (NOUT == 32) {
#pragma unroll
                    for (int c = 0; c < COUT; ++c) y[mt][c] = __uint_as_float(v[c]) + __uint_as_float(v[COUT + c]);
                } else {
#pragma unroll
                    for (int c = 0; c < 32; ++c) y[mt][c % COUT] = __uint_as_float(v[c]);
                    tmem_ld32(taddr + 32, v);
#pragma unroll
                    for (int c = 0; c < 32; ++c) y[mt][c % COUT] += __uint_as_float(v[c]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[buf]);           // accumulators are in registers now
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int m = q * 32 + lane;
                const int aidx = mt * 16 + (m >> 3), hh = m & 7;
                const int d = aidx / 10, w2 = aidx % 10;
                if (d >= D || w2 < 1 || w2 > 8 || (a.dbg & 32)) continue;       // padding columns / junk rows
                if (TRIPLE && row * 3 + d >= n_samples) continue;               // past the last sample
                __align__(16) __nv_bfloat16 hi[COUT], lo[COUT];
#pragma unroll
                for (int c = 0; c < COUT; ++c) {
                    float x = fmaxf(y[mt][c] + sconst[c], 0.f);
                    if (MODE == 1) x = fmaf(x, sconst[COUT + c], sconst[2 * COUT + c]);
                    split2(x, hi[c], lo[c]);
                }
                if (MODE == 0) {
                    // next conv's input, slab order [row][d][w][chunk][h][8]: chunks = hi[0:8] hi[8:16] lo[0:8] lo[8:16]
                    uint4* o = reinterpret_cast<uint4*>(a.out0) +
                               ((((size_t)row * D + d) * 8 + (w2 - 1)) * (2 * COUT / 8)) * 8 + hh;
#pragma unroll
                    for (int i = 0; i < COUT / 8; ++i) o[i * 8] = reinterpret_cast<const uint4*>(hi)[i];
#pragma unroll
                    for (int i = 0; i < COUT / 8; ++i) o[(COUT / 8 + i) * 8] = reinterpret_cast<const uint4*>(lo)[i];
                } else {
                    // dense-1 operand: Keras Flatten order (d, h, w, c)
                    const size_t p = ((size_t)row * D + d) * 64 + hh * 8 + (w2 - 1);
                    uint4* oh = reinterpret_cast<uint4*>(a.out0 + p * COUT);
                    uint4* ol = reinterpret_cast<uint4*>(a.out1 + p * COUT);
#pragma unroll
                    for (int i = 0; i < COUT / 8; ++i) {
                        oh[i] = reinterpret_cast<const uint4*>(hi)[i];
                        ol[i] = reinterpret_cast<const uint4*>(lo)[i];
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<TCOLS>(tmem_base);
    }
}

// =====================================================================================================
// Dense layers: split-bf16 GEMM
// =====================================================================================================
struct GemmTcArgs {
    const int* n_rows;
    const float *bias, *bn_scale, *bn_shift;
    __nv_bfloat16 *out_hi, *out_lo;      // dense 1: next layer's operand [row][N]
    float* out;                          // dense 2: [row][57]
    float* keypoints;                    // dense 2: scatter target or nullptr
    const int32_t *row_scene, *row_slot;
    int K, N, tcap;
    int dbg;                             // timing experiments only (MMW_GEMM_DBG): 1 = no TMA loads, 2 = no MMAs
    float* results = nullptr;            // dense 2, throughput mode: packed result records to finish (pose_tc.cuh)
    const int32_t* row_track = nullptr;
    FadeCfg fade = {0, 0, 0, 0, 0, 0};
};

constexpr int kGemmThreads = 192;
constexpr int kBK = 64;

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}

// Tail of dense 2: the 57 outputs of `nrow` consecutive rows starting at row0 are staged row-major in shared memory
// (stg); 128 epilogue threads (et = 0..127, warp quadrant q) write them out coalesced, scatter them to the tracks'
// keypoint slots and, in throughput mode, finish the packed result records of the frame.  The rows' scene / slot /
// track indices were copied to shared memory (maps: [3][128]) while the main loop ran -- read in the loops below,
// every row would pay an L2 round trip before its stores (32 rows per warp: most of the epilogue's time).
__device__ __forceinline__ void gemm_load_row_maps(const GemmTcArgs& a, int* maps, int row0, int nrow, int et) {
    for (int i = et; i < nrow; i += 128) {
        maps[i] = a.keypoints || a.results ? __ldg(a.row_scene + row0 + i) : 0;
        maps[128 + i] = a.keypoints ? __ldg(a.row_slot + row0 + i) : 0;
        maps[256 + i] = a.results ? __ldg(a.row_track + row0 + i) : 0;
    }
}
__device__ __forceinline__ void gemm_store_keypoints(const GemmTcArgs& a, const float* stg, const int* maps, int row0,
                                                     int nrow, int q, int lane, int et) {
    float* o = a.out + (size_t)row0 * kKp;                             // rows row0.. are contiguous in out
    for (int i = et; i < nrow * kKp; i += 128) o[i] = stg[i];
    if (a.keypoints) {
        for (int r = q; r < nrow; r += 4) {
            float* kp = a.keypoints + ((size_t)maps[r] * a.tcap + maps[128 + r]) * kKp;
            for (int n = lane; n < kKp; n += 32) kp[n] = stg[r * kKp + n];
        }
    }
    if (a.results) {
        for (int r = q; r < nrow; r += 4) {
            float* rec = a.results + ((size_t)maps[r] * a.tcap + maps[256 + r]) * MMW_RESULT_FLOATS;
            for (int n = lane; n < kKp; n += 32) rec[11 + n] = stg[r * kKp + n];
            if (lane == 0) {     // the tracker side left x[0], x[1] as two doubles in rec[68..71]
                const double x0 = reinterpret_cast<const double*>(rec + 68)[0], x1 = reinterpret_cast<const double*>(rec + 68)[1];
                write_fade_square(a.fade, x0, x1, stg + r * kKp, rec);
            }
        }
    }
}

template <int BN, int STAGES>
constexpr int gemm_smem_bytes() { return STAGES * (2 * 128 * kBK * 2 + 2 * BN * kBK * 2) + 1024 + 256 + 3 * 128 * 4; }

// Dense 2 on 128 x BN tiles of one CTA (cta_group::1): out = acc + bias (first 57 columns), scattered to tracks.
// KS > 1: split K over a cluster of KS CTAs (blockIdx.x = cluster rank = K slice).  Dense 2 has only
// ceil(rows / 128) row tiles -- 16 CTAs at C2 -- and each of them streamed 1.1 MB of operands through ONE SM's L2 port
// (14 us of main loop for 0.34 GFLOP).  With the split, KS times as many SMs pull a KS-th each; the partial
// accumulators go TMEM -> registers -> the leader's shared memory (st.shared::cluster into the idle pipeline stages)
// and the leader adds them in rank order: the sum of a row does not depend on where the row sits in the batch.
template <int BN, int STAGES, int KS = 1>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
               const __grid_constant__ CUtensorMap map_wh, const __grid_constant__ CUtensorMap map_wl,
               const GemmTcArgs a) {
    constexpr int BM = 128, UK = 16;
    constexpr int A_BYTES = BM * kBK * 2, B_BYTES = BN * kBK * 2;
    constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr uint32_t TCOLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));   // power of two
    // The row count was written by the feature kernel, at least two kernels upstream: under the PDL discipline
    // (mmw_internal.cuh) that grid had completed before this one could start, so it may be read before pdl_wait()
    // -- which lets the CTAs past the last row leave without holding shared memory while they wait.
    const int rows = __ldcg(a.n_rows);
    const int m0 = blockIdx.y * BM;
    if (m0 >= rows) return;

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ks = KS > 1 ? (int)blockIdx.x : 0;         // cluster rank (cluster = (KS, 1, 1), gridDim.x = KS)
    const int nkb = a.K / kBK / KS, kb0 = ks * nkb;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ah) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_al) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_wh) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_wl) : "memory");
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc<TCOLS>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;
    pdl_wait();                          // the previous layer's activations are complete and visible
    pdl_launch_dependents();

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                unsigned char* st = smem + s * STAGE_BYTES;
                if (a.dbg & 1) { mbar_arrive(&full[s]); continue; }
                mbar_expect_tx(&full[s], STAGE_BYTES);
                const int k0 = (kb0 + kb) * kBK;
                tma_load_2d(st, &map_ah, &full[s], k0, m0);
                tma_load_2d(st + A_BYTES, &map_al, &full[s], k0, m0);
                tma_load_2d(st + 2 * A_BYTES, &map_wh, &full[s], k0, 0);
                tma_load_2d(st + 2 * A_BYTES + B_BYTES, &map_wl, &full[s], k0, 0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(BN);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
                const uint64_t dah = make_desc<128>(st), dal = make_desc<128>(st + A_BYTES);
                const uint64_t dwh = make_desc<128>(st + 2 * A_BYTES), dwl = make_desc<128>(st + 2 * A_BYTES + B_BYTES);
#pragma unroll
                for (int kk = 0; kk < kBK / UK; ++kk) {
                    if (a.dbg & 2) break;
                    const uint64_t adv = (uint64_t)((kk * UK * 2) >> 4);
                    umma_bf16(tmem_d, dah + adv, dwh + adv, idesc, (kb | kk) != 0);
                    umma_bf16(tmem_d, dah + adv, dwl + adv, idesc, 1);
                    umma_bf16(tmem_d, dal + adv, dwh + adv, idesc, 1);
                }
                umma_commit(&empty[s]);
            }
            umma_commit(tmem_full);
        }
    } else if (KS > 1) {
        // accumulators of this K slice into registers; the exchange follows below, outside the role branches
    } else {
        const int q = warp & 3;
        // the rows' scene / slot / track indices into shared memory while the main loop runs
        int* maps = reinterpret_cast<int*>(tmem_slot + 2);
        gemm_load_row_maps(a, maps, m0, min(BM, rows - m0), threadIdx.x - 64);
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        const int row = m0 + q * 32 + lane;
        // the 57 outputs of a row go through shared memory (the pipeline stages are idle now) so that the global writes
        // below are coalesced; lane-per-row scalar stores cost 32 sectors per instruction
        float* stg = reinterpret_cast<float*>(smem);
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            if (row >= rows) continue;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int n = c0 + j;
                if (n < kKp) stg[(q * 32 + lane) * kKp + n] = __uint_as_float(v[j]) + __ldg(a.bias + n);
            }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");                         // the four epilogue warps
        gemm_store_keypoints(a, stg, maps, m0, min(BM, rows - m0), q, lane, threadIdx.x - 64);
    }
    if (KS > 1) {
        // Reduce-scatter by row quadrant: the 32 rows TMEM lane quadrant q holds (epilogue warp with warp % 4 == q)
        // are finished by CTA q of the cluster -- every CTA sends three quadrants of its partial accumulator away,
        // receives three partials of its own quadrant, adds the four in rank order (the sum of a row does not depend on
        // where the row sits in the batch) and writes out 32 rows, so the epilogue is spread over the four SMs too.
        static_assert(KS == 1 || (KS == 4 && BN == 64), "split epilogue: 4 CTAs, 4 row quadrants, 64 columns");
        static_assert(KS == 1 || 32768 + 4 * 8192 <= STAGES * STAGE_BYTES, "partials fit in the pipeline stages");
        const int q = warp & 3;                               // epilogue warps 2..5: TMEM lane quadrant = warp % 4
        const int row0 = m0 + 32 * ks, nrow = max(0, min(32, rows - row0));
        int* maps = reinterpret_cast<int*>(tmem_slot + 2);
        uint32_t v0[32], v1[32];
        if (warp >= 2) {
            gemm_load_row_maps(a, maps, row0, nrow, threadIdx.x - 64);
            mbar_wait(tmem_full, 0);
            tc_fence_after();
            tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16), v0);
            tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + 32u, v1);
            tc_fence_before();
        }
        // every CTA of the cluster has finished its MMAs: the pipeline stages of all four are free to receive partials
        cluster_sync_all();
        // partials in the receiver: [source rank][column group of 4][row of the quadrant][4] floats from byte 32768 on
        // (a warp's 32 rows of one column group are 512 contiguous bytes); the bytes below stay free for the output staging
        float* part = reinterpret_cast<float*>(smem + 32768);
        if (warp >= 2 && q != ks) {
            const uint32_t base = mapa_shared(smem_u32(part + (size_t)ks * 2048 + lane * 4), (uint32_t)q);
#pragma unroll
            for (int g = 0; g < 16; ++g) {
                const uint32_t* v = g < 8 ? v0 : v1;
                const int j = (g & 7) * 4;
                asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(base + (uint32_t)(g * 512)),
                             "r"(v[j]), "r"(v[j + 1]), "r"(v[j + 2]), "r"(v[j + 3])
                             : "memory");
            }
        }
        cluster_sync_all();
        if (warp >= 2) {
            float* stg = reinterpret_cast<float*>(smem);
            if (q == ks) {
                const float4* p4 = reinterpret_cast<const float4*>(part);
#pragma unroll
                for (int g = 0; g < 16; ++g) {
                    const uint32_t* v = g < 8 ? v0 : v1;
                    const int j = (g & 7) * 4;
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int o = 0; o < KS; ++o) {                   // fixed order: K slice 0, 1, 2, 3
                        if (o == ks) {
                            acc[0] += __uint_as_float(v[j]); acc[1] += __uint_as_float(v[j + 1]);
                            acc[2] += __uint_as_float(v[j + 2]); acc[3] += __uint_as_float(v[j + 3]);
                        } else {
                            const float4 t = p4[(size_t)o * 512 + g * 32 + lane];
                            acc[0] += t.x; acc[1] += t.y; acc[2] += t.z; acc[3] += t.w;
                        }
                    }
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int n = g * 4 + e;
                        if (n < kKp) stg[lane * kKp + n] = acc[e] + __ldg(a.bias + n);
                    }
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");                     // the four epilogue warps
            gemm_store_keypoints(a, stg, maps, row0, nrow, q, lane, threadIdx.x - 64);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<TCOLS>(tmem_d);
    }
}

// ---- dense 1 on CTA pairs: tcgen05.mma.cta_group::2 ----------------------------------------------------------
// A single CTA with 128 x 192 tiles keeps only two 80 KB stages in flight, so every K block pays the HBM/L2 round trip
// (per K block: (latency + 80 KB transfer + 1152 MMA cycles) / 2 stages ~ 1950 cycles against 1152 of tensor work).
// A CTA pair (two SMs of one TPC, cluster (2,1,1)) runs ONE 256 x BN MMA per K step: each CTA stages its own 128
// rows of A and only HALF of the W tile (BN/2 rows), the tensor cores exchange the halves.  A stage shrinks to
// 32 KB (A) + 24 KB (W) = 56 KB, so four stages fit and the loads run ~3 K blocks ahead of the tensor core.
//   * both CTAs issue their own TMA loads, all of which complete on the LEADER's full barrier (cta_group::2 form of
//     cp.async.bulk.tensor, barrier address mapped into the leader with mapa)
//   * the leader's elected thread issues every MMA; tcgen05.commit multicasts the "stage free" / "accumulator
//     ready" arrivals to the barriers of both CTAs
//   * each CTA's epilogue warps read the CTA's own TMEM (its 128 rows x BN columns)
// dst in this CTA's shared memory, completion bytes on `bar_cluster` (a shared::cluster address, the leader's barrier)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once the MMAs issued so far have completed) on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                     "r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(COLS) : "memory");
}
// kind::f16 instruction descriptor of the pair MMA: M = 256 (128 rows per CTA)
__device__ __forceinline__ constexpr uint32_t make_idesc_pair(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

template <int BN, int STAGES>
constexpr int gemm_pair_smem_bytes() {
    return STAGES * (2 * 128 * kBK * 2 + 2 * (BN / 2) * kBK * 2) + 1024 + 256 + 3 * BN * 4;
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                    const __grid_constant__ CUtensorMap map_wh_half, const __grid_constant__ CUtensorMap map_wl_half,
                    const GemmTcArgs a) {
    constexpr int BM = 128, UK = 16;
    constexpr int A_BYTES = BM * kBK * 2, BH_BYTES = (BN / 2) * kBK * 2;
    constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * BH_BYTES;              // per CTA
    constexpr uint32_t TCOLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
    __shared__ unsigned long long ts[8];                       // MMW_GEMM_DBG=4: %globaltimer at the phase boundaries
    auto mark = [&](int i) {
        if (a.dbg & 4) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ts[i] = t; }
    };
    if (threadIdx.x == 0) mark(0);
    const int rows = __ldcg(a.n_rows);                         // safe before pdl_wait(): see gemm_tc_kernel
    // grid = (M tiles rounded up to even, N tiles), cluster (2,1,1): a kernel that uses cta_group::2 must pair its CTAs
    // along x (the driver rejects any other cluster shape as "cluster misconfiguration")
    if ((int)(blockIdx.x & ~1u) * BM >= rows) return;          // the whole pair is past the last row
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const uint32_t rank = cluster_ctarank();                   // 0 = leader (issues the MMAs, owns the full barriers)

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* tmem_full = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb = a.K / kBK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ah) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_al) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_wh_half) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_wl_half) : "memory");
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc_pair<TCOLS>(tmem_slot);          // the same warp of both CTAs, collectively
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                        // both CTAs' barriers exist before any remote arrive
    tc_fence_after();
    const uint32_t tmem_d = *tmem_slot;
    pdl_wait();                                                // conv2's output (A_hi / A_lo) is complete and visible
    pdl_launch_dependents();
    if (threadIdx.x == 0) mark(1);

    if (warp == 0) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);                  // own copy: the commit below arrives in both CTAs
                unsigned char* st = smem + s * STAGE_BYTES;
                const uint32_t bar = mapa_shared(smem_u32(&full[s]), 0);
                if (a.dbg & 1) {
                    if (rank == 0) mbar_arrive(&full[s]);
                    continue;
                }
                if (rank == 0) mbar_expect_tx(&full[s], 2 * STAGE_BYTES);       // the bytes of both CTAs
                tma_load_2d_pair(st, &map_ah, bar, kb * kBK, m0);
                tma_load_2d_pair(st + A_BYTES, &map_al, bar, kb * kBK, m0);
                tma_load_2d_pair(st + 2 * A_BYTES, &map_wh_half, bar, kb * kBK, n0 + (int)rank * (BN / 2));
                tma_load_2d_pair(st + 2 * A_BYTES + BH_BYTES, &map_wl_half, bar, kb * kBK, n0 + (int)rank * (BN / 2));
            }
            mark(2);
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc = make_idesc_pair(BN);
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
                const uint64_t dah = make_desc<128>(st), dal = make_desc<128>(st + A_BYTES);
                const uint64_t dwh = make_desc<128>(st + 2 * A_BYTES), dwl = make_desc<128>(st + 2 * A_BYTES + BH_BYTES);
#pragma unroll
                for (int kk = 0; kk < kBK / UK; ++kk) {
                    if (a.dbg & 2) break;
                    const uint64_t adv = (uint64_t)((kk * UK * 2) >> 4);
                    umma_bf16_pair(tmem_d, dah + adv, dwh + adv, idesc, (kb | kk) != 0);
                    umma_bf16_pair(tmem_d, dah + adv, dwl + adv, idesc, 1);
                    umma_bf16_pair(tmem_d, dal + adv, dwh + adv, idesc, 1);
                }
                umma_commit_pair(&empty[s], (uint16_t)3);      // frees the stage in BOTH CTAs
            }
            umma_commit_pair(tmem_full, (uint16_t)3);          // both epilogues may read their accumulators
            mark(3);
        }
    } else {
        const int q = warp & 3;
        // bias / BatchNorm constants of this column tile into shared memory while the main loop runs
        float* sconst = reinterpret_cast<float*>(tmem_slot + 2);
        // (BN need not divide N: the last column tile of the 176-wide variant is 128 wide, its missing W rows come in
        // as zeros from the tensor map's out-of-bounds fill and its missing columns are not stored)
        const int ncols = min(BN, a.N - n0);
        for (int i = threadIdx.x - 64; i < ncols; i += 128) {
            sconst[i] = __ldg(a.bias + n0 + i);
            sconst[BN + i] = __ldg(a.bn_scale + n0 + i);
            sconst[2 * BN + i] = __ldg(a.bn_shift + n0 + i);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        mbar_wait(tmem_full, 0);
        tc_fence_after();
        if (threadIdx.x == 64) mark(4);
        const int row = m0 + q * 32 + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < ncols; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            if (row >= rows) continue;
            const int nv4 = min(32, ncols - c0) >> 3;             // 16-byte vectors of this block that exist (8 columns each)
            __align__(16) __nv_bfloat16 hi[32], lo[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                float x = fmaxf(__uint_as_float(v[j]) + sconst[c0 + j], 0.f);
                x = fmaf(x, sconst[BN + c0 + j], sconst[2 * BN + c0 + j]);
                split2(x, hi[j], lo[j]);
            }
            uint4* oh = reinterpret_cast<uint4*>(a.out_hi + (size_t)row * a.N + n0 + c0);
            uint4* ol = reinterpret_cast<uint4*>(a.out_lo + (size_t)row * a.N + n0 + c0);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (i < nv4) {
                    oh[i] = reinterpret_cast<const uint4*>(hi)[i];
                    ol[i] = reinterpret_cast<const uint4*>(lo)[i];
                }
            }
        }
    }
    if (threadIdx.x == 64) mark(5);
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) mark(6);
    cluster_sync_all();                                        // the peer may still arrive on / read from this CTA
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_pair<TCOLS>(tmem_d);
    }
    if ((a.dbg & 4) && threadIdx.x == 0 && (blockIdx.x < 2 || blockIdx.x == 15) && (blockIdx.y == 0 || blockIdx.y == 7)) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        printf("[pair %d,%d] t0 %llu | prologue %llu | tma issued %llu | mma issued %llu | acc ready %llu | epilogue %llu | "
               "sync %llu | end %llu (ns since t0)\n", (int)blockIdx.x, (int)blockIdx.y, ts[0], ts[1] - ts[0],
               ts[2] - ts[0], ts[3] - ts[0], ts[4] - ts[0], ts[5] - ts[0], ts[6] - ts[0], t - ts[0]);
    }
}

// fp32 feature maps [rows][D*64][5] (position = (d, h, w)) -> packed bf16 in slab order [rows][D][8 w][2][8 h][8]:
// chunk 0 = (hi c0..4, 0,0,0), chunk 1 = (lo c0..4, 0,0,0)
__global__ void pack_input_kernel(const float* __restrict__ feats, __nv_bfloat16* __restrict__ out, const int* n_rows,
                                  int P) {
    const size_t total = (size_t)(*n_rows) * P;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        __align__(16) __nv_bfloat16 v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = __float2bfloat16_rn(0.f);
#pragma unroll
        for (int k = 0; k < 5; ++k) split2(feats[i * 5 + k], v[k], v[8 + k]);
        const size_t slice = i / 64;                       // row * D + d
        const int pos = (int)(i % 64), h = pos >> 3, w = pos & 7;
        uint4* o = reinterpret_cast<uint4*>(out) + ((slice * 8 + w) * 2) * 8 + h;
        o[0] = reinterpret_cast<const uint4*>(v)[0];
        o[8] = reinterpret_cast<const uint4*>(v)[1];
    }
}

// ---- host side ---------------------------------------------------------------------------------------
struct TcImpl {
    int D = 0, taps = 0, Kf = 0, H = 0, rows_cap = 0, rows_pad = 0;
    __nv_bfloat16 *in_p = nullptr, *in_p2 = nullptr, *act1_p = nullptr;   // packed activations (input double-buffered)
    __nv_bfloat16 *a_hi = nullptr, *a_lo = nullptr;                   // dense-1 operand [rows_pad][Kf]
    __nv_bfloat16 *h_hi = nullptr, *h_lo = nullptr;                   // dense-2 operand [rows_pad][H]
    __nv_bfloat16 *w1b = nullptr, *w2b = nullptr;                     // conv B matrices [taps][NOUT][CK]
    __nv_bfloat16 *wd1_hi = nullptr, *wd1_lo = nullptr, *wd2_hi = nullptr, *wd2_lo = nullptr;
    CUtensorMap m_w1b, m_w2b, m_ah, m_al, m_hh, m_hl, m_w2h, m_w2l;
    // dense-1 W halves (BN / 2 rows) of the pair kernels by tile width; 176 and 192 only when 192 divides H
    CUtensorMap m_w1h_half256, m_w1l_half256, m_w1h_half192, m_w1l_half192, m_w1h_half176, m_w1l_half176;
    int force_bn = 0;                                                 // MMW_FC1_BN = 176 / 192 / 256 (tests)
    int pair_slots = 74;                                              // CTA pairs that run at once (SMs / 2)
    int dbg = 0;
};

static std::string g_tc_err;
const char* pose_tc_error() { return g_tc_err.c_str(); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}

static CUtensorMapSwizzle swz(int bytes) {
    return bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// 2-D bf16 tensor [rows][K] (K contiguous), box [box_rows][box_k], swizzle span = box_k * 2 bytes.
static int make_map_2d(CUtensorMap* m, void* base, uint64_t rows, uint64_t K, uint32_t box_rows, uint32_t box_k) {
    EncodeTiledFn enc = get_encode();
    if (!enc) { g_tc_err = "cuTensorMapEncodeTiled not available"; return -1; }
    cuuint64_t dims[2] = {K, rows};
    cuuint64_t strides[1] = {K * 2};
    cuuint32_t box[2] = {box_k, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swz((int)box_k * 2), CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_tc_err = "cuTensorMapEncodeTiled(2d) failed (" + std::to_string((int)r) + ")"; return -1; }
    return 0;
}

static inline uint16_t f2bf(float f) {            // round-to-nearest-even, like __float2bfloat16_rn
    uint32_t u;
    std::memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static inline float bf2f(uint16_t h) {
    uint32_t u = (uint32_t)h << 16;
    float f;
    std::memcpy(&f, &u, 4);
    return f;
}

template <class T>
static bool dev_alloc(T** p, size_t bytes, bool zero = false) {
    if (cudaMalloc((void**)p, bytes) != cudaSuccess) return false;
    if (zero) cudaMemset(*p, 0, bytes);
    return true;
}
static bool upload(__nv_bfloat16** d, const std::vector<uint16_t>& h) {
    if (!dev_alloc(d, h.size() * 2)) return false;
    return cudaMemcpy(*d, h.data(), h.size() * 2, cudaMemcpyHostToDevice) == cudaSuccess;
}

// Conv B operand of one layer: [taps][2*cout][2*cinp] (K-major rows):
//   n <  cout : k <  cinp -> w_hi[k][n]        k >= cinp -> w_hi[k-cinp][n]
//   n >= cout : k <  cinp -> w_lo[k][n-cout]   k >= cinp -> 0
// w is Keras layout [tap][cin][cout]; input channels are zero-padded from cin to cinp.
static std::vector<uint16_t> conv_b(const float* w, int taps, int cin, int cinp, int cout) {
    const int CK = 2 * cinp, NO = 2 * cout;
    std::vector<uint16_t> b((size_t)taps * NO * CK, 0);
    for (int t = 0; t < taps; ++t)
        for (int n = 0; n < NO; ++n)
            for (int k = 0; k < CK; ++k) {
                const int ci = k % cinp, co = n % cout;
                if (ci >= cin) continue;
                const float wv = w[((size_t)t * cin + ci) * cout + co];
                const uint16_t hi = f2bf(wv), lo = f2bf(wv - bf2f(hi));
                uint16_t v = 0;
                if (n < cout) v = hi;
                else if (k < cinp) v = lo;
                b[((size_t)t * NO + n) * CK + k] = v;
            }
    return b;
}

// Conv 2 B operand: [taps][3 cout][cin] (one K16 per row): rows 0..cout-1 w_hi, cout..2cout-1 w_lo (both for the a_hi
// chunk), 2cout..3cout-1 w_hi again (for the a_lo chunk).  cin must be 16.
static std::vector<uint16_t> conv_b2(const float* w, int taps, int cin, int cout) {
    std::vector<uint16_t> b((size_t)taps * 3 * cout * cin, 0);
    for (int t = 0; t < taps; ++t)
        for (int r = 0; r < 3 * cout; ++r)
            for (int ci = 0; ci < cin; ++ci) {
                const int co = r % cout;
                const float wv = w[((size_t)t * cin + ci) * cout + co];
                const uint16_t hi = f2bf(wv), lo = f2bf(wv - bf2f(hi));
                b[((size_t)t * 3 * cout + r) * cin + ci] = (r >= cout && r < 2 * cout) ? lo : hi;
            }
    return b;
}

// Dense weight [K][N] (Keras in,out) -> K-major [Npad][K] hi / lo.
static void dense_b(const float* w, int K, int N, int Npad, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
    hi.assign((size_t)Npad * K, 0);
    lo.assign((size_t)Npad * K, 0);
    for (int k = 0; k < K; ++k)
        for (int n = 0; n < N; ++n) {
            const float wv = w[(size_t)k * N + n];
            const uint16_t h = f2bf(wv);
            hi[(size_t)n * K + k] = h;
            lo[(size_t)n * K + k] = f2bf(wv - bf2f(h));
        }
}

int pose_tc_init(PoseTc* t, const float* blob, const size_t* off, int D, int rows_cap) {
    pose_tc_free(t);
    TcImpl* im = new TcImpl();
    t->impl = im;
    im->D = D; im->taps = D == 3 ? 27 : 9; im->Kf = D * 64 * 32; im->H = D * 512; im->rows_cap = rows_cap;
    im->rows_pad = (rows_cap + 127) / 128 * 128;
    t->D = D; t->K = im->Kf; t->H = im->H; t->rows_cap = rows_cap;
    const size_t R = im->rows_pad, P = (size_t)D * 64;
    bool ok = dev_alloc(&im->in_p, R * P * 16 * 2, true) && dev_alloc(&im->in_p2, R * P * 16 * 2, true) &&
              dev_alloc(&im->act1_p, R * P * 32 * 2, true) &&
              dev_alloc(&im->a_hi, R * im->Kf * 2, true) && dev_alloc(&im->a_lo, R * im->Kf * 2, true) &&
              dev_alloc(&im->h_hi, R * im->H * 2, true) && dev_alloc(&im->h_lo, R * im->H * 2, true);
    { const char* env = getenv("MMW_GEMM_DBG"); im->dbg = env ? atoi(env) : 0; }
    if (!ok) { g_tc_err = "cudaMalloc failed (activations)"; return -1; }
    std::vector<uint16_t> hi, lo;
    ok = upload(&im->w1b, conv_b(blob + off[0], im->taps, 5, 8, 16)) &&
         upload(&im->w2b, conv_b2(blob + off[2], im->taps, 16, 32));
    dense_b(blob + off[8], im->Kf, im->H, im->H, hi, lo);
    ok = ok && upload(&im->wd1_hi, hi) && upload(&im->wd1_lo, lo);
    dense_b(blob + off[14], im->H, kKp, 64, hi, lo);
    ok = ok && upload(&im->wd2_hi, hi) && upload(&im->wd2_lo, lo);
    if (!ok) { g_tc_err = "cudaMalloc/cudaMemcpy failed (weights)"; return -1; }
    if (make_map_2d(&im->m_w1b, im->w1b, (uint64_t)im->taps * 32, 16, 32, 16) ||
        make_map_2d(&im->m_w2b, im->w2b, (uint64_t)im->taps * 96, 16, 96, 16) ||
        make_map_2d(&im->m_ah, im->a_hi, R, im->Kf, 128, 64) || make_map_2d(&im->m_al, im->a_lo, R, im->Kf, 128, 64) ||
        make_map_2d(&im->m_w1h_half256, im->wd1_hi, im->H, im->Kf, 128, 64) ||
        make_map_2d(&im->m_w1l_half256, im->wd1_lo, im->H, im->Kf, 128, 64) ||
        make_map_2d(&im->m_hh, im->h_hi, R, im->H, 128, 64) || make_map_2d(&im->m_hl, im->h_lo, R, im->H, 128, 64) ||
        make_map_2d(&im->m_w2h, im->wd2_hi, 64, im->H, 64, 64) || make_map_2d(&im->m_w2l, im->wd2_lo, 64, im->H, 64, 64))
        return -1;
    cudaError_t e = cudaSuccess;
    auto set_smem = [&](const void* fn, int bytes) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        // every kernel of the step asks for the same (maximum) shared-memory carve-out, so the SMs are not
        // reconfigured at each of the seven kernel boundaries of a step
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    };
    set_smem((const void*)conv_slab_kernel<16, 32, 0, 3>, conv_smem_bytes_tc<16, 32>(27));
    set_smem((const void*)conv_slab_kernel<32, 64, 1, 3>, conv_smem_bytes_tc<32, 64>(27));
    set_smem((const void*)conv_slab_kernel<16, 32, 0, 1>, conv_smem_bytes_tc<16, 32>(9));
    set_smem((const void*)conv_slab_kernel<32, 64, 1, 1>, conv_smem_bytes_tc<32, 64>(9));
    set_smem((const void*)gemm_tc_kernel<64, 4>, gemm_smem_bytes<64, 4>());
    set_smem((const void*)gemm_tc_kernel<64, 4, 4>, gemm_smem_bytes<64, 4>());
    if (e != cudaSuccess) { g_tc_err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return -1; }
    // Dense 1 on CTA pairs with three pipeline stages (four were measured too: no faster than three, the main loop
    // already runs at the tensor-core floor).  Whether a 2-CTA cluster of every tile width the launcher may pick can
    // run on this device is asked of the driver, not assumed (on a B200 all three fit: <= 201 KB of shared memory);
    // a kernel that cannot be scheduled fails the initialisation.
    auto pair_fits = [&](const void* fn, int bytes, int bn) -> bool {
        set_smem(fn, bytes);
        int n = 0;
        if (e == cudaSuccess) {
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(2, 8);
            cfg.blockDim = dim3(kGemmThreads);
            cfg.dynamicSmemBytes = bytes;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            e = cudaOccupancyMaxActiveClusters(&n, fn, &cfg);
        }
        const std::string name = "gemm_tc_pair_kernel<" + std::to_string(bn) + ",3>";
        if (e != cudaSuccess) {
            (void)cudaGetLastError();     // not left behind for the next launch check to report
            g_tc_err = name + ": " + cudaGetErrorString(e);
            return false;
        }
        if (n < 1) {
            g_tc_err = name + ": a cluster of two CTAs with " + std::to_string(bytes) +
                       " bytes of shared memory each cannot be scheduled on this device";
            return false;
        }
        return true;
    };
    // 256 x 192 tiles need ceil(rows / 256) * 8 CTA pairs: one wave up to 2304 rows (74 pairs on 148 SMs), two
    // beyond -- twice the time for one row more.  256 x 256 tiles (6 per row block, 4/3 of the time each) stay in one
    // wave up to 3072 rows, 256 x 176 tiles (9 per row block, the last one 128 wide) up to 2048 rows at 11/12 of the
    // time; the launcher takes whichever is cheapest for the row count of an earlier frame.  The 2-D net (H = 512)
    // always uses 256-wide tiles.
    if (!pair_fits((const void*)gemm_tc_pair_kernel<256, 3>, gemm_pair_smem_bytes<256, 3>(), 256)) return -1;
    if (im->H % 192 == 0) {
        if (!pair_fits((const void*)gemm_tc_pair_kernel<192, 3>, gemm_pair_smem_bytes<192, 3>(), 192) ||
            !pair_fits((const void*)gemm_tc_pair_kernel<176, 3>, gemm_pair_smem_bytes<176, 3>(), 176))
            return -1;
        if (make_map_2d(&im->m_w1h_half192, im->wd1_hi, im->H, im->Kf, 96, 64) ||
            make_map_2d(&im->m_w1l_half192, im->wd1_lo, im->H, im->Kf, 96, 64) ||
            make_map_2d(&im->m_w1h_half176, im->wd1_hi, im->H, im->Kf, 88, 64) ||
            make_map_2d(&im->m_w1l_half176, im->wd1_lo, im->H, im->Kf, 88, 64))
            return -1;
    }
    {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        im->pair_slots = sms / 2;
    }
    { const char* benv = getenv("MMW_FC1_BN"); im->force_bn = benv ? atoi(benv) : 0; }
    t->ready = true;
    return 0;
}

__nv_bfloat16* pose_tc_input(PoseTc* t, int buf) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    return im ? (buf ? im->in_p2 : im->in_p) : nullptr;
}

static int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { g_tc_err = std::string(what) + ": " + cudaGetErrorString(e); return -1; }
    return 0;
}

int pose_tc_pack_input(PoseTc* t, const float* feats, const int* n_rows, cudaStream_t st) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (!im || !t->ready) { g_tc_err = "tensor-core path not initialised"; return -1; }
    pack_input_kernel<<<148 * 4, 256, 0, st>>>(feats, im->in_p, n_rows, im->D * 64);
    return check_launch("pack_input_kernel");
}

int pose_tc_conv(PoseTc* t, const PoseTcRun& r, cudaStream_t st, int* n_launches, int buf) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (!im || !t->ready) { g_tc_err = "tensor-core path not initialised"; return -1; }
    // the 2-D net (KD = 1) runs three samples per slab
    ConvTcArgs c1{r.n_rows, r.b1, nullptr, nullptr, buf ? im->in_p2 : im->in_p, im->act1_p, nullptr, im->dbg};
    const dim3 one(1, 1, 1);
    cudaError_t le;
    if (im->D == 3)
        le = launch_pdl(conv_slab_kernel<16, 32, 0, 3>, dim3(148), dim3(kSlabThreads), conv_smem_bytes_tc<16, 32>(27), st, one,
                        im->m_w1b, c1);
    else
        le = launch_pdl(conv_slab_kernel<16, 32, 0, 1>, dim3(148), dim3(kSlabThreads), conv_smem_bytes_tc<16, 32>(9), st, one,
                        im->m_w1b, c1);
    if (le != cudaSuccess) { g_tc_err = std::string("conv_slab_kernel<conv1>: ") + cudaGetErrorString(le); return -1; }
    ConvTcArgs c2{r.n_rows, r.b2, r.bn1_scale, r.bn1_shift, im->act1_p, im->a_hi, im->a_lo, im->dbg};
    if (im->D == 3)
        le = launch_pdl(conv_slab_kernel<32, 64, 1, 3>, dim3(148), dim3(kSlabThreads), conv_smem_bytes_tc<32, 64>(27), st, one,
                        im->m_w2b, c2);
    else
        le = launch_pdl(conv_slab_kernel<32, 64, 1, 1>, dim3(148), dim3(kSlabThreads), conv_smem_bytes_tc<32, 64>(9), st, one,
                        im->m_w2b, c2);
    if (le != cudaSuccess) { g_tc_err = std::string("conv_slab_kernel<conv2>: ") + cudaGetErrorString(le); return -1; }
    if (n_launches) *n_launches = 2;
    return 0;
}

int pose_tc_fc1(PoseTc* t, const PoseTcRun& r, int max_rows, cudaStream_t st, int* n_launches, int rows_hint) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (!im || !t->ready) { g_tc_err = "tensor-core path not initialised"; return -1; }
    GemmTcArgs g{r.n_rows, r.bd1, r.bn2_scale, r.bn2_shift, im->h_hi, im->h_lo, nullptr, nullptr, nullptr, nullptr,
                 im->Kf, im->H, r.tcap, im->dbg};
    int bn = 256;
    if (im->H % 192 == 0) {
        bn = 192;
        if (rows_hint > 0) {
            // cost of a launch = waves of CTA pairs x tile width; 176 (9 column tiles), 192 (8) or 256 (6) columns
            // (the hint is a frame or two old and the row count drifts by a few rows per frame: plan for 48 more -- one row
            // past a tile-count edge costs a whole second wave)
            const int mt = (rows_hint + 48 + 255) / 256, P = im->pair_slots;
            auto cost = [&](int w) { return ((mt * ((im->H + w - 1) / w) + P - 1) / P) * w; };
            int best = cost(192);
            if (cost(256) < best) { best = cost(256); bn = 256; }
            if (cost(176) < best) bn = 176;
        }
        if (im->force_bn == 176 || im->force_bn == 192 || im->force_bn == 256) bn = im->force_bn;
    }
    const dim3 grid((((max_rows + 127) / 128) + 1) & ~1, (im->H + bn - 1) / bn), blk(kGemmThreads), cl(2, 1, 1);
    cudaError_t le;
    if (bn == 176)
        le = launch_pdl(gemm_tc_pair_kernel<176, 3>, grid, blk, gemm_pair_smem_bytes<176, 3>(), st, cl, im->m_ah, im->m_al,
                        im->m_w1h_half176, im->m_w1l_half176, g);
    else if (bn == 192)
        le = launch_pdl(gemm_tc_pair_kernel<192, 3>, grid, blk, gemm_pair_smem_bytes<192, 3>(), st, cl, im->m_ah, im->m_al,
                        im->m_w1h_half192, im->m_w1l_half192, g);
    else
        le = launch_pdl(gemm_tc_pair_kernel<256, 3>, grid, blk, gemm_pair_smem_bytes<256, 3>(), st, cl, im->m_ah, im->m_al,
                        im->m_w1h_half256, im->m_w1l_half256, g);
    if (le != cudaSuccess) { g_tc_err = std::string("dense 1 launch: ") + cudaGetErrorString(le); return -1; }
    if (n_launches) *n_launches = 1;
    return 0;
}

int pose_tc_fc2(PoseTc* t, const PoseTcRun& r, int max_rows, cudaStream_t st, int* n_launches) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (!im || !t->ready) { g_tc_err = "tensor-core path not initialised"; return -1; }
    GemmTcArgs g{r.n_rows, r.bd2, nullptr, nullptr, nullptr, nullptr, r.out, r.keypoints, r.row_scene, r.row_slot,
                 im->H, 64, r.tcap, im->dbg, r.results, r.row_track, r.fade};
    // K split over a cluster of 4 CTAs per row tile whenever the K blocks divide (1536 / 64 = 24, 512 / 64 = 8)
    cudaError_t le;
    if ((im->H / kBK) % 4 == 0 && (max_rows + 127) / 128 <= 128)      // large batches fill the SMs without it
        le = launch_pdl(gemm_tc_kernel<64, 4, 4>, dim3(4, (max_rows + 127) / 128), dim3(kGemmThreads),
                        gemm_smem_bytes<64, 4>(), st, dim3(4, 1, 1), im->m_hh, im->m_hl, im->m_w2h, im->m_w2l, g);
    else
        le = launch_pdl(gemm_tc_kernel<64, 4>, dim3(1, (max_rows + 127) / 128), dim3(kGemmThreads),
                        gemm_smem_bytes<64, 4>(), st, dim3(1, 1, 1), im->m_hh, im->m_hl, im->m_w2h, im->m_w2l, g);
    if (le != cudaSuccess) { g_tc_err = std::string("dense 2 launch: ") + cudaGetErrorString(le); return -1; }
    if (n_launches) *n_launches = 1;
    return 0;
}

int pose_tc_intermediate(PoseTc* t, int layer, int n, uint16_t* out) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (!im || !t->ready) { g_tc_err = "tensor-core path not initialised"; return -1; }
    const size_t P = (size_t)im->D * 64, rows = (size_t)n;
    const size_t per = layer == 0 ? P * 5 : layer == 1 ? P * 16 : layer == 2 ? (size_t)im->Kf : (size_t)im->H;
    uint16_t* lo_out = out + rows * per;
    if (layer >= 2) {
        const __nv_bfloat16* src[2] = {layer == 2 ? im->a_hi : im->h_hi, layer == 2 ? im->a_lo : im->h_lo};
        for (int p = 0; p < 2; ++p)
            if (cudaMemcpy(p ? lo_out : out, src[p], rows * per * 2, cudaMemcpyDeviceToHost) != cudaSuccess) {
                g_tc_err = "cudaMemcpy (intermediate)";
                return -1;
            }
        return 0;
    }
    // slab order [row][d][w][chunk][h][8]: the input has chunks (hi c0..4 | lo c0..4), conv 1's output
    // (hi c0..7, hi c8..15, lo c0..7, lo c8..15)
    const int nch = layer == 0 ? 2 : 4, cout = layer == 0 ? 5 : 16;
    std::vector<uint16_t> h(rows * P * nch * 8);
    if (cudaMemcpy(h.data(), layer == 0 ? im->in_p : im->act1_p, h.size() * 2, cudaMemcpyDeviceToHost) != cudaSuccess) {
        g_tc_err = "cudaMemcpy (intermediate)";
        return -1;
    }
    for (size_t r = 0; r < rows; ++r)
        for (size_t pos = 0; pos < P; ++pos) {
            const size_t d = pos / 64, hh = (pos / 8) % 8, w = pos % 8;
            const size_t base = ((r * im->D + d) * 8 + w) * nch;
            for (int c = 0; c < cout; ++c) {
                const int chunk_hi = c / 8, chunk_lo = nch / 2 + c / 8;
                const size_t o = (r * P + pos) * cout + c;
                out[o] = h[((base + chunk_hi) * 8 + hh) * 8 + c % 8];
                lo_out[o] = h[((base + chunk_lo) * 8 + hh) * 8 + c % 8];
            }
        }
    return 0;
}

void pose_tc_free(PoseTc* t) {
    TcImpl* im = reinterpret_cast<TcImpl*>(t->impl);
    if (im) {
        for (void* p : {(void*)im->in_p, (void*)im->in_p2, (void*)im->act1_p, (void*)im->a_hi, (void*)im->a_lo, (void*)im->h_hi,
                        (void*)im->h_lo, (void*)im->w1b, (void*)im->w2b, (void*)im->wd1_hi, (void*)im->wd1_lo,
                        (void*)im->wd2_hi, (void*)im->wd2_lo})
            if (p) cudaFree(p);
        delete im;
    }
    t->impl = nullptr;
    t->ready = false;
}

}  // namespace mmw
