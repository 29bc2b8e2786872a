// Block-cooperative exact-neighbourhood DBSCAN with sklearn's canonical labelling
// (Utils.apply_DBscan, Utils.py:250-291; sklearn DBSCAN.fit + dbscan_inner; SURVEY Appendix A Q1-Q6).
//
//   neighbourhood(p) = { q : altered_EuclideanDist(p, q) <= eps }, p included
//   core(p)          = |neighbourhood(p)| >= min_samples
//   clusters         = connected components of the core-core epsilon graph (union-find, smaller index is
//                      the root, so the root is the smallest core index of the component)
//   label(core p)    = rank of its root among all roots in ascending index order
//   label(border p)  = min label over core points within eps, else -1 (noise)
//
// which is exactly what dbscan_inner's ascending outer loop + DFS produces.
#pragma once
#include <cmath>
#include "mmw_internal.cuh"

namespace mmw {

// Find with path halving.  Parents only ever decrease (roots are hooked under smaller roots), so shortening a path
// with atomicMin(parent, grandparent) can never undo a concurrent hook -- a plain store could.  Without it the
// min-index hooking degenerates into linked lists and every find in a dense 100-point blob walks ~100 links.
__device__ __forceinline__ int uf_find(int* par, int i) {
    while (true) {
        const int p = ((volatile int*)par)[i];
        if (p == i) return i;
        const int gp = ((volatile int*)par)[p];
        if (gp != p) atomicMin(&par[i], gp);
        i = p;
    }
}

__device__ __forceinline__ void uf_unite(int* par, int a, int b) {
    while (true) {
        a = uf_find(par, a);
        b = uf_find(par, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }   // hook the larger root under the smaller
        const int old = atomicMin(&par[a], b);
        if (old == a) return;
        a = old;                                          // a had already been hooked elsewhere: merge that too
    }
}

// Exclusive block scan of one flag per thread; returns this thread's rank, *total = number of set flags.
// s_scan: blockDim.x/32 + 1 ints of shared memory.  Must be called by every thread of the block.
__device__ __forceinline__ int block_rank(bool flag, int* total, int* s_scan) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_scan[warp] = __popc(m);
    __syncthreads();
    int before = 0, tot = 0;
    for (int w = 0; w < nw; ++w) {
        const int c = s_scan[w];
        if (w < warp) before += c;
        tot += c;
    }
    __syncthreads();
    *total = tot;
    return before + __popc(m & ((1u << lane) - 1u));
}

// Neighbour predicates ------------------------------------------------------------------------------------
// Exact: float64 world coordinates in shared memory (stage-level entry point mmw_dbscan).
struct NbExact {
    const DevConfig& c;
    const double *X, *Y, *Z;
    double eps;
    __device__ __forceinline__ bool operator()(int b, int q) const {
        return eps_neighbour(c, X[b], Y[b], Z[b], X[q], Y[q], Z[q], eps);
    }
    __device__ __forceinline__ const NbExact& hot() const { return *this; }
};

// Screened: the fused step keeps the world coordinates of the ring points rounded to fp32 in shared memory and
// evaluates the predicate in fp32 first (FP32 pipe, 4-cycle ops); only pairs whose fp32 distance falls inside a
// guard band around eps -- wider than any fp32 rounding could move it -- are re-evaluated exactly in float64 from
// the raw ring rows.  Decisions are therefore identical to the exact predicate, at a fraction of the FP64 work
// (the FP64/XU pipe is what bounds this kernel, profiles/).
//
// The band only covers the fp32 error where that error is bounded, so the screen has a domain: |y'|, |z'| <= R.
// A point outside it gets Xf = NaN (screen_domain_mark), which makes the fp32 distance of every pair it is in NaN:
// such a pair is neither above hi nor below lo and goes to float64.  Derivation (u = 2^-24, first order in u; rw, zw
// >= 0; both points inside the domain, so w = 1 - rw (y1 + y2) / 2 lies in [w_min, 2] with w_min = 1 - rw R):
//   inputs   x exact, Yf = y (1 + d), |d| <= u, same for Zf; rw and zw rounded to fp32 (relative u)
//   w        |w_f - w| <= 4 u rw R + u |w_f| <= 6 u
//   q        dx^2 + dy^2 + zw dz^2: 7 u q from the roundings of the products and sums (all terms >= 0), plus the
//            rounding of the inputs, |dy_f - dy| <= 2 u R + u |dy|, which adds 4 u R |dy| <= 4 u R sqrt(q), and
//            4 u R zw |dz| <= 4 u R sqrt(zw q) for the z term
//   d = w q  |d_f - d| <= |w_f - w| q + |w| |q_f - q| + u |d_f| <= 22 u q + 8 u R sqrt(q) (1 + sqrt(zw))
// Fused multiply-adds only remove roundings, so the bound holds for any contraction.  A pair decided wrongly has
// d <= eps < hi < d_f or d_f < lo < eps < d, so q <= (eps + band) / w_min (1 + O(u)) =: Q / 2.  R is chosen
// (screen_config) so that the bound at Q is at most half the band; the other half covers the fp32 rounding of eps,
// lo and hi (~u eps, the band is >= 1e-3 eps) and the float64 rounding of the exact predicate.  w_min is 0.25
// (R <= 0.75 / rw): the band would need to grow as 1 / w near w = 0, where the fp32 error does.
// tests/dbscan_screen_model.py restates this function and screen_config.
__device__ __forceinline__ float screen_d(float xb, float yb, float zb, float xq, float yq, float zq, float rw,
                                          float zw) {
    const float w = 1.f - 0.5f * (yb + yq) * rw;
    const float dx = xb - xq, dy = yb - yq, dz = zb - zq;
    return w * (dx * dx + dy * dy + zw * (dz * dz));
}

// The fp32 x of a point as the screen stores it: NaN outside the screen's domain (every pair of the point goes to
// float64, see screen_d).  yw, zw: the point's float64 world coordinates.
__device__ __forceinline__ float screen_domain_mark(float x, double yw, double zw, float rmax) {
    return fabs(yw) <= (double)rmax && fabs(zw) <= (double)rmax ? x : __int_as_float(0x7fc00000);
}

// Host side: guard band and domain radius for a configuration (mmw_create).  rmax = -1 (every pair exact): eps not
// positive and finite, a negative or non-finite weight, or no radius at which the bound holds.
inline void screen_config(double eps, double range_weight, double z_weight, float* lo, float* hi, float* rmax) {
    const float band = 1e-3f * (float)eps + 1e-4f;
    *lo = (float)eps - band;
    *hi = (float)eps + band;
    *rmax = -1.f;
    if (!(eps > 0.0 && eps < 1e30) || !(range_weight >= 0.0 && range_weight < 1e30) ||
        !(z_weight >= 0.0 && z_weight < 1e30))
        return;
    const double u = 0x1p-24, wmin = 0.25;
    const double Q = 2.0 * (eps + (double)band) / wmin;
    double R = (0.5 * (double)band - 22.0 * u * Q) / (8.0 * u * std::sqrt(Q) * (1.0 + std::sqrt(z_weight)));
    if (range_weight > 0.0) R = std::fmin(R, (1.0 - wmin) / range_weight);
    if (!(R > 0.0)) return;
    R = std::fmin(R, 1e30);
    float r = (float)R;
    if ((double)r > R) r = std::nextafter(r, 0.f);                   // round down
    *rmax = r;
}

struct NbScreened {
    const DevConfig& c;
    const SensorRec& sr;              // the scene's mounting (shared memory)
    const float *Xf, *Yf, *Zf;        // shared memory, B floats each
    const float* frame[kRing];        // raw rows of the ring frames, oldest first (global)
    int start[kRing + 1];             // first fused index of each frame
    double eps;
    float lo, hi, rw, zw;
    const float* rawc;                // the same raw rows in fused order in shared memory, or nullptr (dbscan_big_kernel)
    __device__ __forceinline__ void world(int b, double& x, double& y, double& z) const {
        const int f = (b >= start[1] ? 1 : 0) + (b >= start[2] ? 1 : 0);
        const float* r = rawc != nullptr ? rawc + (size_t)b * kRawCols : frame[f] + (size_t)(b - start[f]) * kRawCols;
        x = (double)r[0];
        world_yz(sr, (double)r[1], (double)r[2], y, z);
    }
    // out of line on purpose: its float64 registers must not be live across the fp32 hot loop
    __device__ __noinline__ bool exact(int b, int q) const {
        double x1, y1, z1, x2, y2, z2;
        world(b, x1, y1, z1);
        world(q, x2, y2, z2);
        return eps_neighbour(c, x1, y1, z1, x2, y2, z2, eps);
    }
    // The part of the predicate that runs for every pair, as a small by-value functor: seven scalars that stay in
    // registers (the full struct has indexed arrays and lives in local memory -- going through it cost ~300 cycles
    // per pair in LDL traffic).
    struct Hot {
        const float *X, *Y, *Z;
        float lo, hi, rw, zw;
        const NbScreened* full;
        __device__ __forceinline__ bool operator()(int b, int q) const {
            const float d = screen_d(X[b], Y[b], Z[b], X[q], Y[q], Z[q], rw, zw);
            if (d > hi) return false;
            if (d < lo) return true;
            return full->exact(b, q);                   // inside the guard band or outside the domain: decide exactly
        }
    };
    __device__ __forceinline__ Hot hot() const { return Hot{Xf, Yf, Zf, lo, hi, rw, zw, this}; }
};

// Conservative screen "can any point of the fused ring be a core point?" on a fixed 16 x 16 grid over the world
// (x, y') plane.  Two points within eps of each other satisfy dx^2 + dy^2 <= eps / w with
// w = 1 - range_weight (y1 + y2)/2 >= 1 - range_weight * ybound for y' <= ybound (Utils.py:242-247; the z term only
// adds), so with cells at least sqrt(eps / w_min) wide every neighbour of a point lies in the 3 x 3 block of cells
// around it: if no block around an occupied cell holds min_samples points, no point has min_samples neighbours and
// DBSCAN labels everything noise -- which is what the steady-state residue of ~70 clutter points does in > 99.9 %
// of the scene-frames (tests/test_grid_screen_cpu.py).  Cells outside the grid are folded onto its border (counts
// can only grow).  Because the cells do not depend on the cloud, every ring frame is binned ONCE, when it is pushed
// (the points are in registers then), and kept as 256 saturating byte counts + a flag byte per frame next to the
// ring (StepArgs::ring_hist); the screen itself is a sum of three small histograms and 256 box sums -- no point is
// touched again.  The flag marks a frame with a point beyond ybound (or not finite): then the screen passes.
constexpr int kGridDim = 16, kGridCells = kGridDim * kGridDim;

// Host side: cell size and validity for a configuration (mmw_create).  ybound: 12 m covers every radar profile of
// the reference (config_cases/*.cfg: <= 8.5 m) and keeps w_min at 0.64 for the default range weight.
inline void grid_screen_config(double eps, double range_weight, double z_weight, int min_samples, float* inv_h,
                               float* ybound, int* ok) {
    *ok = 0; *inv_h = 0.f; *ybound = 0.f;
    if (!(range_weight >= 0.0) || !(z_weight >= 0.0) || !(eps > 0.0) || min_samples > 255) return;
    double yb = 12.0;
    if (range_weight * yb > 0.5) yb = 0.5 / range_weight;              // keep w_min >= 0.5
    const float wmin = 1.f - (float)range_weight * ((float)yb * 1.0001f);
    if (!(wmin > 0.05f)) return;
    const float h = 1.01f * sqrtf((float)eps / wmin);                  // 1 % wider than the largest xy reach
    *inv_h = 1.f / h;
    *ybound = (float)yb;
    *ok = 1;
}

__device__ __forceinline__ int grid_cell(const DevConfig& c, float x, float yw) {
    const int kx = (int)floorf(x * c.grid_inv_h + 0.5f * kGridDim), ky = (int)floorf(yw * c.grid_inv_h);
    const int cx = kx < 0 ? 0 : (kx >= kGridDim ? kGridDim - 1 : kx);
    const int cy = ky < 0 ? 0 : (ky >= kGridDim ? kGridDim - 1 : ky);
    return cy * kGridDim + cx;
}

// sum[cell]: points of the fused ring per cell (shared memory).  Returns the same value in every thread of the
// block; false means "certainly no core point".  Ends with a block barrier.
__device__ __forceinline__ bool grid_screen_may_have_core(const uint16_t* sum, int min_samples) {
    int cand = 0;
    for (int cell = threadIdx.x; cell < kGridCells; cell += blockDim.x) {
        if (sum[cell] == 0) continue;
        const int cx = cell % kGridDim, cy = cell / kGridDim;
        int n = 0;
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int x = cx + dx, y = cy + dy;
                if (x >= 0 && x < kGridDim && y >= 0 && y < kGridDim) n += sum[y * kGridDim + x];
            }
        cand |= n >= min_samples ? 1 : 0;
    }
    return __syncthreads_or(cand) != 0;
}

// par, cl: B ints each (shared).  On return cl[b] is the label of b.
// Returns the number of clusters (uniform over the block).
// Sweep over all unordered pairs q < b < B in warp tiles: a warp owns a chunk of 32 consecutive q (one per lane) and
// walks the rows b above it, so one row step evaluates 32 pairs, the row side of a result is combined with a warp
// ballot / shuffle and the column side stays in a lane register.  fn(b, q, live) is called by all 32 lanes
// (live = this lane's pair exists).
template <class Fn>
__device__ __forceinline__ void for_pair_tiles(int B, Fn fn) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int nchunk = (B + 31) >> 5;
    // every warp visits every chunk and takes the rows b = first + warp, first + warp + nw, ... : the work of a
    // chunk (long for low j, short for high j) is split evenly instead of landing on one warp
    for (int j = 0; j < nchunk; ++j) {
        const int q = (j << 5) + lane;
        for (int b = (j << 5) + 1 + warp; b < B; b += nw) fn(b, q, q < b && q < B);
    }
}

constexpr unsigned kFullMask = 0xffffffffu;

template <class Nb>
// stop_if_core: return -1 right after the counts when any core point exists (the caller hands the scene to
// dbscan_big_kernel: clusters form in a couple of scenes per frame and the remaining sweeps would make that CTA
// the one the whole step kernel waits for).
__device__ inline int dbscan_block(const Nb& nb_full, int B, int min_samples, int* par, int* cl, int* s_scan,
                                   unsigned long long* dbg = nullptr, bool stop_if_core = false,
                                   bool dbg_border = false) {
    const auto nb = nb_full.hot();
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    long long dbg_t = clock64();
    auto stamp = [&](int k) {
        if (dbg != nullptr && tid == 0) {
            const long long now = clock64();
            atomicAdd(&dbg[k], (unsigned long long)(now - dbg_t));
            dbg_t = now;
        }
    };
    // 1. neighbour counts: |{q : d(p,q) <= eps}| including p.  One integer atomic per (row, chunk) with a hit and
    //    one per lane and chunk -- order-independent, so the counts (and everything below) are deterministic.
    //    (Register-resident 32 x 32 tiles of the upper triangle, as in dbscan_bits_block, were measured here too:
    //    slower with the step kernel's four warps -- 18.9 k against 15.4 k cycles per scene-frame.)
    for (int b = tid; b < B; b += nt) par[b] = 1;                      // a point is its own neighbour
    __syncthreads();
    {
        int cq = 0, qprev = -1;
        for_pair_tiles(B, [&](int b, int q, bool live) {
            if (q != qprev) {                                           // new chunk: flush this lane's column count
                if (cq) atomicAdd(&par[qprev], cq);
                cq = 0; qprev = q;
            }
            const bool hit = live && nb(b, q);
            const unsigned m = __ballot_sync(kFullMask, hit);
            cq += hit ? 1 : 0;
            if (lane == 0 && m) atomicAdd(&par[b], __popc(m));
        });
        if (cq) atomicAdd(&par[qprev], cq);
    }
    __syncthreads();
    stamp(13);
    int anycore = 0;
    for (int b = tid; b < B; b += nt) {
        const bool core = par[b] >= min_samples;
        par[b] = core ? b : -1;
        anycore |= core ? 1 : 0;
    }
    anycore = __syncthreads_or(anycore);
    if (!anycore) {
        for (int b = tid; b < B; b += nt) cl[b] = -1;
        __syncthreads();
        return 0;
    }
    if (stop_if_core) return -1;
    // 2. connected components over core points (par[x] >= 0 <=> x is core, stable under the unions).  Pairs that
    //    are already in one component are skipped BEFORE the predicate is evaluated: inside a dense blob almost
    //    every pair is.
    for_pair_tiles(B, [&](int b, int q, bool live) {
        if (((volatile int*)par)[b] < 0) return;                        // uniform over the warp
        if (!live || ((volatile int*)par)[q] < 0) return;
        if (uf_find(par, q) == uf_find(par, b)) return;
        if (nb(b, q)) uf_unite(par, b, q);
    });
    __syncthreads();
    stamp(14);
    for (int b = tid; b < B; b += nt) cl[b] = par[b] >= 0 ? uf_find(par, b) : -1;
    __syncthreads();
    // rank of each root among the roots, ascending index
    int ncl = 0;
    for (int base = 0; base < B; base += nt) {
        const int b = base + tid;
        const bool isroot = b < B && cl[b] == b;
        int tot;
        const int r = block_rank(isroot, &tot, s_scan);
        if (isroot) par[b] = ncl + r;          // par[root] now holds the cluster id
        ncl += tot;
    }
    __syncthreads();
    for (int b = tid; b < B; b += nt) {
        const int r = cl[b];
        if (r >= 0) cl[b] = par[r];
    }
    __syncthreads();
    stamp(15);
    // 3. border points: lowest-numbered cluster with a core point within eps (cl[x] >= 0 <=> x is core here)
    for (int b = tid; b < B; b += nt)
        if (cl[b] < 0) par[b] = 0x7fffffff;
    __syncthreads();
    for_pair_tiles(B, [&](int b, int q, bool live) {
        const int lb = cl[b];                                           // uniform over the warp
        const int lq = live ? cl[q] : lb;
        const bool mixed = live && ((lb >= 0) != (lq >= 0));
        const bool hit = mixed && nb(b, q);
        if (lb >= 0) {                                                  // core row: label flows to non-core lanes
            if (hit) atomicMin(&par[q], lb);
        } else {                                                        // non-core row: min label of the core lanes
            int v = hit ? lq : 0x7fffffff;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(kFullMask, v, o));
            if (lane == 0 && v != 0x7fffffff) atomicMin(&par[b], v);
        }
    });
    __syncthreads();
    for (int b = tid; b < B; b += nt)
        if (cl[b] < 0) cl[b] = par[b] == 0x7fffffff ? -1 : par[b];
    __syncthreads();
    if (dbg_border) stamp(16);
    return ncl;
}

// ---------------------------------------------------------------------------------------------------------
// The same DBSCAN on an explicit adjacency bit matrix (dbscan_big_kernel).  The pair sweeps above evaluate the
// predicate up to three times per pair and are chained through shared-memory atomics; for the handful of scenes per
// frame in which clusters actually form that chain IS the kernel's duration.  Here the predicate is evaluated once
// per unordered pair into adj[b][w] (bit j of word w = point 32 w + j is within eps of b, b included), and everything
// after that is word-wide bit arithmetic:
//   counts      popc of a row; core mask cm by ballot
//   components  frontier expansion on bit masks: start from the lowest core point not yet visited -- the point
//               dbscan_inner's ascending scan starts a cluster from, so clusters come out in canonical order --
//               and OR the core rows of the frontier into the component until it stops growing (a person-sized blob
//               is a near-clique: two rounds)
//   border      a non-core point takes the first (= lowest-numbered) cluster whose mask meets its row
// Results are independent of scheduling (integer ORs only).  Shared memory: adj B * W words, cm W words,
// ws (4 + kMaxCompMasks) * W words, W = ceil(B / 32).  Requires B <= blockDim.x * 32 and W <= blockDim.x.
constexpr int kMaxCompMasks = 32;      // clusters whose masks are kept for the border step (more: row-pull fallback)

__device__ inline int dbscan_bits_block(const NbScreened& nbf, int B, int min_samples, unsigned* adj, unsigned* cm,
                                        unsigned* ws, int* /*par*/, int* cl, unsigned long long* dbg = nullptr) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int W = (B + 31) >> 5;
    unsigned *visited = ws, *comp = ws + W, *front = ws + 2 * W, *next = ws + 3 * W, *cmask = ws + 4 * W;
    long long dbg_t = clock64();
    auto stamp = [&](int k) {
        if (dbg != nullptr && tid == 0) {
            const long long now = clock64();
            atomicAdd(&dbg[k], (unsigned long long)(now - dbg_t));
            dbg_t = now;
        }
    };
    // 1. adjacency rows, by 32 x 32 tiles of the upper triangle (the predicate is symmetric): a warp owns tile (I, J),
    //    I <= J; lane = column q of word J with its coordinates in registers, the 32 rows b of block I are broadcast
    //    from shared memory.  A row step gives word adj[b][J] by ballot; each lane collects its own hits over the rows,
    //    which is the transposed word adj[q][I].  The fp32 screen decides almost every pair, the few inside the guard
    //    band are settled exactly (same decisions as NbScreened::Hot, see there).
    {
        const float *X = nbf.Xf, *Y = nbf.Yf, *Z = nbf.Zf;
        const float lo = nbf.lo, hi = nbf.hi, rw = nbf.rw, zw = nbf.zw;
        const int ntiles = W * (W + 1) / 2;
        for (int t = warp; t < ntiles; t += nw) {
            int I = 0, rem = t;
            while (rem >= W - I) { rem -= W - I; ++I; }
            const int J = I + rem;
            const int q = (J << 5) + lane;
            const bool qlive = q < B;
            const float xq = qlive ? X[q] : 0.f, yq = qlive ? Y[q] : 0.f, zq = qlive ? Z[q] : 0.f;
            const int b0 = I << 5, bn = min(32, B - b0);
            unsigned tb = 0;
            // two rows per step: their dependent chains (broadcast loads -> distance -> ballot) overlap
            for (int r = 0; r < bn; r += 2) {
                const int ba = b0 + r, bb = r + 1 < bn ? ba + 1 : ba;
                const float da = screen_d(X[ba], Y[ba], Z[ba], xq, yq, zq, rw, zw);
                const float db = screen_d(X[bb], Y[bb], Z[bb], xq, yq, zq, rw, zw);
                bool hita = qlive && (da < lo || q == ba), hitb = qlive && (db < lo || q == bb);
                // in the band or outside the screen's domain (NaN)
                const bool unsa = qlive && !(da > hi) && !hita, unsb = qlive && !(db > hi) && !hitb;
                if (__any_sync(kFullMask, unsa || unsb)) {
                    if (unsa) hita = nbf.exact(ba, q);
                    if (unsb) hitb = nbf.exact(bb, q);
                }
                const unsigned ma = __ballot_sync(kFullMask, hita), mb = __ballot_sync(kFullMask, hitb);
                if (lane == 0) {
                    adj[ba * W + J] = ma;
                    if (bb != ba) adj[bb * W + J] = mb;
                }
                tb |= (hita ? 1u : 0u) << r;
                if (bb != ba) tb |= (hitb ? 1u : 0u) << (r + 1);
            }
            if (I != J && qlive) adj[q * W + I] = tb;
        }
    }
    __syncthreads();
    // neighbour counts -> core mask (one warp per word of points)
    for (int w = warp; w < W; w += nw) {
        const int b = (w << 5) + lane;
        int cnt = 0;
        if (b < B)
            for (int ww = 0; ww < W; ++ww) cnt += __popc(adj[b * W + ww]);
        const unsigned m = __ballot_sync(kFullMask, b < B && cnt >= min_samples);
        if (lane == 0) { cm[w] = m; visited[w] = 0u; next[w] = 0u; }
    }
    for (int b = tid; b < B; b += nt) cl[b] = -1;
    __syncthreads();
    stamp(13);
    // 2. components of the core-core graph, in ascending order of their lowest core point
    int ncl = 0;
    while (true) {
        int L = -1;
        for (int w = 0; w < W; ++w) {
            const unsigned u = cm[w] & ~visited[w];
            if (u) { L = (w << 5) + __ffs(u) - 1; break; }
        }
        if (L < 0) break;                                               // uniform over the block
        if (tid < W) comp[tid] = front[tid] = tid == (L >> 5) ? 1u << (L & 31) : 0u;
        __syncthreads();
        while (true) {
            for (int b0 = warp << 5; b0 < B; b0 += nt) {
                const int b = b0 + lane;
                const bool in_front = b < B && ((front[b >> 5] >> (b & 31)) & 1u);
                if (!__any_sync(kFullMask, in_front)) continue;
                for (int w = 0; w < W; ++w) {
                    const unsigned v = __reduce_or_sync(kFullMask, in_front ? (adj[b * W + w] & cm[w]) : 0u);
                    if (lane == 0 && v) atomicOr(&next[w], v);
                }
            }
            __syncthreads();
            int grew = 0;
            if (tid < W) {
                const unsigned fresh = next[tid] & ~comp[tid];
                comp[tid] |= fresh;
                front[tid] = fresh;
                next[tid] = 0u;
                grew = fresh != 0u;
            }
            if (!__syncthreads_or(grew)) break;
        }
        for (int b = tid; b < B; b += nt)
            if ((comp[b >> 5] >> (b & 31)) & 1u) cl[b] = ncl;
        if (tid < W) {
            visited[tid] |= comp[tid];
            if (ncl < kMaxCompMasks) cmask[ncl * W + tid] = comp[tid];
        }
        ++ncl;
        __syncthreads();
    }
    stamp(15);
    // 3. border points: lowest-numbered cluster with a core point within eps
    if (ncl <= kMaxCompMasks) {
        for (int b = tid; b < B; b += nt) {
            if ((cm[b >> 5] >> (b & 31)) & 1u) continue;
            for (int k = 0; k < ncl; ++k) {
                unsigned any = 0u;
                for (int w = 0; w < W; ++w) any |= adj[b * W + w] & cmask[k * W + w];
                if (any) { cl[b] = k; break; }
            }
        }
    } else {                           // more clusters than kept masks: pull the minimum id over the core neighbours
        for (int b = warp; b < B; b += nw) {
            if ((cm[b >> 5] >> (b & 31)) & 1u) continue;                 // uniform over the warp
            int m = 0x7fffffff;
            for (int w = 0; w < W; ++w) {
                const unsigned bits = adj[b * W + w] & cm[w];
                if ((bits >> lane) & 1u) m = min(m, cl[(w << 5) + lane]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(kFullMask, m, o));
            __syncwarp();
            if (lane == 0 && m != 0x7fffffff) cl[b] = m;
        }
    }
    __syncthreads();
    stamp(16);
    return ncl;
}

}  // namespace mmw
