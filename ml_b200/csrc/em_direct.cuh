// Gaussian-mixture EM, direct-difference kernels: any K, D <= 128, and every shape whose components sit far from the
// centre of the data in their own standard deviations.
//
// The feature-space kernels (em.cu, em_small.cuh, em_split.cuh) evaluate the quadratic form about ONE shift c (the data
// mean): q = -1/2 z^T P z + z^T P delta - 1/2 delta^T P delta with z = x - c, delta = mu_k - c, and take the covariance as
// m2/s - (m1/s)(m1/s)^T.  Both cancel by kappa_k = delta^T P_k delta: harmless for standardised data (kappa ~ 1e2..1e3,
// error ~1e-13), not for tight clusters thousands of standard deviations apart (kappa = 1e8 costs 8 digits).  The
// reference has no such term: it evaluates (x - mu_k)^T P_k (x - mu_k) directly (ML/EM.cpp:205-207,
// LinearAlgebra.cpp:8-31) and accumulates the covariance about the new mean (EM.cpp:246-248).  These kernels do the
// same per component, still on the FP64 tensor pipe:
//
//   E kernel  y = P'_k w,  w = z - delta_k, as a [points x D] x [D x D] DMMA product over the 8 x 8 blocks of the upper
//             block triangle (P' = P on the diagonal blocks, 2 P above them: the symmetric form LinearAlgebra.cpp:17-29
//             sums), then q = w . y in the accumulator layout; the component images stream through a cp.async double
//             buffer; log-densities go to R[point][KPr], a half-warp per point does the log-sum-exp in place.
//   M kernel  per component the augmented second moment sum_i r_ik [w, 1][w, 1]^T about the component's OLD mean
//             (SURVEY.md H3), upper block triangle, as [D+8 x points] x [points x D+8] DMMA products; the new mean is
//             mu_old + m1/s and the covariance m2/s - (m1/s)(m1/s)^T, whose cancellation is |mu_new - mu_old|^2 / sigma^2
//             and vanishes as the fit converges.  r w and w are staged per component in shared memory.
// Work per point-component pair: E D^2 + D, M (D + 8)^2 / 2 + ... multiply-adds, i.e. about twice the feature path; this
// path runs when the feature path is out of its domain (em_finalize_kernel reports kappa, the host routes), for D > 64
// or K > 256, and on request (mlb_em_force_path).
//
// Statistics are written per SUPER-CHUNK (a run of consecutive chunks of one virtual shard, a function of N only), not
// per chunk: a component's statistics are (NB + 1)(NB + 2)/2 tiles of 64 doubles (1.5 MB per vector at D = 64, K = 64).
#pragma once

#include "em_split.cuh"
#include "fastmath.cuh"
#include "internal.h"

namespace mlb {

constexpr int kDrTile = 64;       // points per E-step tile (4 warps x 16)
constexpr int kDrThreads = 128;
constexpr int kDrSub = 16;        // points per M-step staging step
constexpr int kDrSlots = 16;      // (component, tile) accumulators per warp of the M kernel
constexpr int kDrSuperPerVshard = 48;   // at most this many super-chunks per virtual shard

__host__ __device__ constexpr int dr_steps(int NB) { return NB * (NB + 1); }                       // DMMA steps of one component's E image
__host__ __device__ constexpr int dr_img_len(int DP) { return dr_steps(DP / 8) * 32 + DP + 8; }    // steps | delta (DP) | log c, padding
__host__ __device__ constexpr int dr_tiles(int NB) { return (NB + 1) * (NB + 2) / 2; }             // tiles of the augmented upper block triangle
__host__ __device__ constexpr int dr_stat_len(int DP) { return dr_tiles(DP / 8) * 64; }
// index of tile (mt <= nt) in the row-major upper triangle over NBa = NB + 1 blocks
__host__ __device__ inline int dr_tile_index(int NBa, int mt, int nt) { return mt * NBa - mt * (mt - 1) / 2 + (nt - mt); }

struct EmDirectArgs {
    const double* x;        // local points, d doubles each
    long long n_local;
    int d, k, DP, KPr;      // DP: D padded to 8; KPr: row stride of R (K padded to 8)
    const double* shift;    // d
    const double* img;      // [k][dr_img_len(DP)] component images (em_finalize_kernel)
    double* r;              // [n_local][KPr]
    double* ll_tile;        // [ceil(n_local / 64)] log-likelihood sum of every E tile; scoring: [n_local] log p(x) of every point
    unsigned* counter;
    int cb;                 // E: components per staged batch
    // M
    const long long* sc_begin;   // [n_sc + 1] local point boundaries of the super-chunks
    int n_sc;
    double* partials;       // [n_sc][svd]: k blocks of dr_stat_len(DP) doubles, then the log-likelihood sum and padding
    int svd;
    int cg;                 // M: components per work item
    int tiles_per_range;    // M: tiles of a component per work item
    int n_ranges;           // M: work items per component group
    const int2* tile_tab;   // [dr_tiles] (mt, nt)
    int unit_r;             // 1: responsibilities are 1 for component 0 and 0 elsewhere (sample covariance); r is not read
};

inline size_t em_direct_e_smem(int DP, int cb)
{
    return sizeof(double) * (static_cast<size_t>(kDrTile) * (DP + 4) + 2 * static_cast<size_t>(cb) * dr_img_len(DP) + DP + kExpTableSize + 8 + kDrTile * 8);
}
inline size_t em_direct_m_smem(int DP, int cg, int d)
{
    return sizeof(double) * ((2 * static_cast<size_t>(cg) + 1) * kDrSub * (DP + 12) + static_cast<size_t>(cg) * DP + DP + 2 * static_cast<size_t>(kDrSub) * (d + (d & 1)) + 2 * static_cast<size_t>(kDrSub) * cg);
}

// ---------------------------------------------------------------- E kernel (expectation_step, EM.cpp:190-219)
// NBT: the number of 8-coordinate blocks when it is 1 or 2 (D <= 16: the loops over the blocks unroll completely), 0 for any D.
// NBTS = NBT, or NBT + kDrScore for the scoring pass, which writes log p(x) per point to ll_tile instead of responsibilities
// and tile sums (r receives the log-densities only).  The flag rides in the one int parameter so that the step's instances
// keep their names and their code.
constexpr int kDrScore = 16;
template <int NBTS>
__global__ void __launch_bounds__(kDrThreads) em_direct_e_kernel(const EmDirectArgs p)
{
    constexpr int NBT = NBTS & (kDrScore - 1);
    constexpr bool SCORE = (NBTS & kDrScore) != 0;
    extern __shared__ __align__(16) double sm[];
    const int DP = NBT ? 8 * NBT : p.DP, NB = DP / 8, ZS = DP + 4, IMG = dr_img_len(DP), SPC = dr_steps(NB), d = p.d;
    double* Z = sm;                                     // [64][ZS]
    double* buf = Z + kDrTile * ZS;                     // [2][cb * IMG]
    double* sh = buf + 2 * static_cast<size_t>(p.cb) * IMG;   // [DP]
    double* etab = sh + DP;                             // [32]
    double* wl = etab + kExpTableSize;                  // [8]
    double* Qs = wl + 8;                                // [4 warps][16 points][8 components]: log-densities on their way to R
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    double* Qw = Qs + warp * (16 * 8);
    for (int i = tid; i < kDrTile * ZS; i += kDrThreads) Z[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    load_exp_table(etab);

    const int nbatches = (p.k + p.cb - 1) / p.cb;
    auto stage = [&](int b, int which) {
        const int k0 = b * p.cb, nc = min(p.cb, p.k - k0);
        const double* src = p.img + static_cast<size_t>(k0) * IMG;
        double* dst = buf + static_cast<size_t>(which) * p.cb * IMG;
        for (int i = tid; i < nc * IMG / 2; i += kDrThreads) sp_cp_async16(dst + 2 * i, src + 2 * i);
        sp_cp_async_commit();
    };

    const int ntiles = static_cast<int>((p.n_local + kDrTile - 1) / kDrTile);
    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int item = s_next;
        if (item >= ntiles) break;
        const long long tile0 = static_cast<long long>(item) * kDrTile;
        const int nvalid = static_cast<int>(p.n_local - tile0 < kDrTile ? p.n_local - tile0 : kDrTile);
        sp_load_z_tile(Z, ZS, p.x, sh, tile0, nvalid, d, DP);   // z = x - c; column DP holds a constant the kernel never reads
        const double* z0 = Z + (warp * 16 + g) * ZS;
        const double* z1 = z0 + 8 * ZS;
        // a lane pair flushes one point's 8 staged log-densities as a 64-byte segment of its R row
        const int fp = lane >> 1, fh = (lane & 1) * 4;
        double* frow = p.r + (tile0 + warp * 16 + fp) * p.KPr + fh;
        const bool flive = warp * 16 + fp < nvalid;

        stage(0, 0);
        for (int b = 0; b < nbatches; ++b) {
            if (b + 1 < nbatches) {
                stage(b + 1, (b + 1) & 1);
                sp_cp_async_wait<1>();
            } else {
                sp_cp_async_wait<0>();
            }
            __syncthreads();   // the batch (and, for b == 0, the point tile) is visible
            const int k0 = b * p.cb, nc = min(p.cb, p.k - k0);
            const double* base = buf + static_cast<size_t>(b & 1) * p.cb * IMG;
            for (int kk = 0; kk < nc; ++kk) {
                const double* im = base + static_cast<size_t>(kk) * IMG;
                const double* dl = im + SPC * 32;
                double q0 = 0.0, q1 = 0.0;
                int step = 0;
#pragma unroll
                for (int B = 0; B < (NBT ? NBT : NB); ++B) {
                    double acc0[2] = {0.0, 0.0}, acc1[2] = {0.0, 0.0};
#pragma unroll 2
                    for (int s2 = 0; s2 < 2 * (B + 1); ++s2, ++step) {
                        const int a = 4 * s2 + c;
                        const double m = dl[a];
                        const double bf = im[step * 32 + lane];
                        sp_dmma(acc0, z0[a] - m, bf);
                        sp_dmma(acc1, z1[a] - m, bf);
                    }
                    const int n0 = 8 * B + 2 * c;
                    const double2 mm = *reinterpret_cast<const double2*>(dl + n0);
                    const double2 u0 = *reinterpret_cast<const double2*>(z0 + n0);
                    const double2 u1 = *reinterpret_cast<const double2*>(z1 + n0);
                    q0 = fma(acc0[0], u0.x - mm.x, fma(acc0[1], u0.y - mm.y, q0));
                    q1 = fma(acc1[0], u1.x - mm.x, fma(acc1[1], u1.y - mm.y, q1));
                }
                q0 += __shfl_xor_sync(0xffffffffu, q0, 1);
                q0 += __shfl_xor_sync(0xffffffffu, q0, 2);
                q1 += __shfl_xor_sync(0xffffffffu, q1, 1);
                q1 += __shfl_xor_sync(0xffffffffu, q1, 2);
                const double logc = dl[DP];
                const int slot = (k0 + kk) & 7;
                if (c == 0) {
                    Qw[g * 8 + slot] = fma(-0.5, q0, logc);
                    Qw[(g + 8) * 8 + slot] = fma(-0.5, q1, logc);
                }
                if (slot == 7 || k0 + kk + 1 == p.k) {
                    // components past K in the last group of 8 are padding: -inf, i.e. responsibility 0
                    __syncwarp();
                    const int kbase = (k0 + kk) & ~7;
                    if (flive) {
                        double v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) v[u] = kbase + fh + u < p.k ? Qw[fp * 8 + fh + u] : -INFINITY;
                        *reinterpret_cast<double2*>(frow + kbase) = make_double2(v[0], v[1]);
                        *reinterpret_cast<double2*>(frow + kbase + 2) = make_double2(v[2], v[3]);
                    }
                    __syncwarp();
                }
            }
            __syncthreads();   // the buffer is refilled two batches later
        }
        // ---------------- log-sum-exp in place: a half-warp per point, 8 passes over the warp's 16 points
        __threadfence_block();
        __syncwarp();
        double ll_acc = 0.0, ll_prod = 1.0;
        const int hl = lane & 15;
        for (int pass = 0; pass < 8; ++pass) {
            const int pl = warp * 16 + pass * 2 + (lane >> 4);
            double* rrow = p.r + (tile0 + pl) * p.KPr;
            const bool live = pl < nvalid;
            double mx = -INFINITY;
            if (live)
                for (int kk = hl; kk < p.k; kk += 16) mx = fmax(mx, __ldcg(rrow + kk));
#pragma unroll
            for (int off = 8; off >= 1; off >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
            double sum = 0.0;
            if (live)
                for (int kk = hl; kk < p.k; kk += 16) sum += exp_nonpositive(__ldcg(rrow + kk) - mx, etab);
#pragma unroll
            for (int off = 8; off >= 1; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
            if constexpr (SCORE) {
                if (live && hl == 0) p.ll_tile[tile0 + pl] = (mx + log(sum)) - 0.5 * d * kLog2Pi;
            } else if (live) {
                const double inv = reciprocal_of_sum(sum);
                for (int kk = hl; kk < p.KPr; kk += 16) rrow[kk] = exp_nonpositive(__ldcg(rrow + kk) - mx, etab) * inv;   // padding: exp(-inf) = 0
                if (hl == 0) {
                    ll_acc += mx;
                    ll_prod *= sum;
                }
            }
        }
        if constexpr (SCORE) {
            __syncthreads();   // Z is rewritten by the next item
            continue;
        }
        ll_acc += log(ll_prod);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) ll_acc += __shfl_xor_sync(0xffffffffu, ll_acc, off);
        if (lane == 0) wl[warp] = ll_acc;
        __syncthreads();   // also: Z is rewritten by the next item
        if (tid == 0) p.ll_tile[item] = (wl[0] + wl[1]) + (wl[2] + wl[3]);
    }
}

// The log-likelihood partial of every super-chunk: its E tiles' sums in a fixed order (lane-strided, then a butterfly).
// One warp per super-chunk.
__global__ void em_direct_ll_kernel(const EmDirectArgs p)
{
    const int sc = blockIdx.x, lane = threadIdx.x;
    const long long t0 = p.sc_begin[sc] / kDrTile, t1 = (p.sc_begin[sc + 1] + kDrTile - 1) / kDrTile;
    double acc = 0.0;
    for (long long t = t0 + lane; t < t1; t += 32) acc += p.ll_tile[t];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    double* out = p.partials + static_cast<long long>(sc) * p.svd + static_cast<long long>(p.k) * dr_stat_len(p.DP);
    if (lane < 8) out[lane] = lane == 0 ? acc : 0.0;
}

// ---------------------------------------------------------------- M kernel (maximisation_step, EM.cpp:221-263)
// Work item = (super-chunk, group of cg components, range of tiles_per_range tiles): cg * tiles_per_range <= 4 * kDrSlots
// (component, tile) pairs, kDrSlots per warp, accumulated in registers over the points of the super-chunk.  The points and
// the responsibilities of the next 16-point sub-tile arrive by cp.async while the current one is multiplied.
__global__ void __launch_bounds__(kDrThreads) em_direct_m_kernel(const EmDirectArgs p)
{
    extern __shared__ __align__(16) double sm[];
    const int DP = p.DP, NB = DP / 8, WS = DP + 12, WSZ = kDrSub * WS, IMG = dr_img_len(DP), SPC = dr_steps(NB), d = p.d, cg = p.cg;
    const int T = dr_tiles(NB), L = dr_stat_len(DP), XSZ = kDrSub * (d + (d & 1)), RSZ = kDrSub * cg;
    double* W = sm;                                    // [cg][16][WS]: w = z - delta_k | 1 | zeros
    double* RW = W + static_cast<size_t>(p.cg) * WSZ;  // [cg + 1][16][WS]: r_ik times the same; the last block is all zeros
    double* dl = RW + static_cast<size_t>(p.cg + 1) * WSZ; // [cg][DP]
    double* sh = dl + static_cast<size_t>(p.cg) * DP;  // [DP]
    double* Xs = sh + DP;                              // [2][16 * d] raw coordinates of a sub-tile, as in global memory
    double* Rs = Xs + 2 * XSZ;                         // [2][16][cg] responsibilities of a sub-tile
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    // Accumulator slots without a (component, tile) pair multiply the zero block: every warp issues the same kDrSlots products
    // per step with no branch around any of them (a branch per slot cost ten times the products it skipped).
    for (int i = tid; i < WSZ; i += kDrThreads) RW[static_cast<size_t>(p.cg) * WSZ + i] = 0.0;

    const int ngroups = (p.k + p.cg - 1) / p.cg;
    const int per_sc = ngroups * p.n_ranges;
    const long long nitems = static_cast<long long>(p.n_sc) * per_sc;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int item = s_next;
        if (item >= nitems) break;
        // consecutive items share a super-chunk, so concurrently running CTAs re-read the same points from L2
        const int sc = item / per_sc, rem = item - sc * per_sc;
        const int grp = rem / p.n_ranges, range = rem - grp * p.n_ranges;
        const int k0 = grp * p.cg, nc = min(p.cg, p.k - k0);
        const int t0 = range * p.tiles_per_range, ntr = min(p.tiles_per_range, T - t0);
        const int npairs = nc * ntr;

        unsigned off[kDrSlots];   // RW offset of the A operand | W offset of the B operand << 16 (both < 2^15 doubles)
        double acc[kDrSlots][2];
#pragma unroll
        for (int t = 0; t < kDrSlots; ++t) {
            const int pair = warp * kDrSlots + t;
            acc[t][0] = acc[t][1] = 0.0;
            unsigned oa = static_cast<unsigned>(p.cg * WSZ + g), ob = static_cast<unsigned>(g);   // the zero block
            if (pair < npairs) {
                const int cl = pair / ntr, tile = t0 + (pair - cl * ntr);
                const int2 mn = p.tile_tab[tile];
                oa = static_cast<unsigned>(cl * WSZ + 8 * mn.x + g);
                ob = static_cast<unsigned>(cl * WSZ + 8 * mn.y + g);
            }
            off[t] = oa | (ob << 16);
        }
        for (int i = tid; i < nc * DP; i += kDrThreads) {
            const int cl = i / DP, a = i - cl * DP;
            dl[i] = p.img[static_cast<size_t>(k0 + cl) * IMG + SPC * 32 + a];
        }
        const long long p_begin = p.sc_begin[sc], p_end = p.sc_begin[sc + 1];
        const int nsubs = static_cast<int>((p_end - p_begin + kDrSub - 1) / kDrSub);
        auto sub_valid = [&](int s) { const long long left = p_end - (p_begin + static_cast<long long>(s) * kDrSub); return static_cast<int>(left < kDrSub ? left : kDrSub); };
        // asynchronous copy of sub-tile s: its coordinates (one contiguous run) and its cg responsibilities per point;
        // rows past the end of the super-chunk get zero coordinates and zero responsibilities (r = 0 removes them from
        // every product, and 0 * w must not meet an Inf or NaN left behind in the buffer)
        auto prefetch = [&](int s, int which) {
            const long long sub0 = p_begin + static_cast<long long>(s) * kDrSub;
            const int nv = sub_valid(s), nel = nv * d;
            const double* xg = p.x + sub0 * d;
            double* xs = Xs + which * XSZ;
            if ((d & 1) == 0) {
                for (int e2 = tid; 2 * e2 < kDrSub * d; e2 += kDrThreads) {
                    if (2 * e2 < nel) sp_cp_async16(xs + 2 * e2, xg + 2 * e2);
                    else *reinterpret_cast<double2*>(xs + 2 * e2) = make_double2(0.0, 0.0);
                }
            } else {
                for (int e = tid; e < kDrSub * d; e += kDrThreads) {
                    if (e < nel) sp_cp_async8(xs + e, xg + e);
                    else xs[e] = 0.0;
                }
            }
            double* rs = Rs + which * RSZ;
            for (int pt = warp; pt < kDrSub; pt += 4)
                for (int cl = lane; cl < nc; cl += 32) {
                    if (p.unit_r) rs[pt * cg + cl] = (pt < nv && k0 + cl == 0) ? 1.0 : 0.0;
                    else if (pt < nv) sp_cp_async8(rs + pt * cg + cl, p.r + (sub0 + pt) * p.KPr + k0 + cl);
                    else rs[pt * cg + cl] = 0.0;
                }
            sp_cp_async_commit();
        };
        if (nsubs > 0) prefetch(0, 0);
        const int CW = DP + 8;                 // coordinates of an augmented row: w | 1 | zeros
        const FastDiv by_cw(CW);
        for (int s = 0; s < nsubs; ++s) {
            if (s + 1 < nsubs) {
                prefetch(s + 1, (s + 1) & 1);
                sp_cp_async_wait<1>();
            } else {
                sp_cp_async_wait<0>();
            }
            __syncthreads();   // sub-tile s has arrived; every warp is past the products of sub-tile s - 1 (first pass: dl, sh)
            const double* xs = Xs + (s & 1) * XSZ;
            const double* rs = Rs + (s & 1) * RSZ;
            // w and r w: a thread takes one (point, coordinate) cell at a time and walks the components, so that the point's
            // coordinate is read and shifted once and the inner loop is two loads, two FP64 operations and two stores
            for (int q = tid; q < kDrSub * CW; q += kDrThreads) {
                const int pt = by_cw.div(q), co = q - pt * CW;
                const bool coord = co < d;
                const double z = coord ? xs[pt * d + co] - sh[co] : (co == DP ? 1.0 : 0.0);
                const double* dlp = dl + (coord ? co : 0);
                const double* rp = rs + pt * cg;
                double* wp = W + pt * WS + co;
                double* rwp = RW + pt * WS + co;
#pragma unroll 2
                for (int cl = 0; cl < nc; ++cl) {
                    const double w = coord ? z - dlp[cl * DP] : z;
                    wp[cl * WSZ] = w;
                    rwp[cl * WSZ] = rp[cl] * w;
                }
            }
            __syncthreads();
#pragma unroll
            for (int s4 = 0; s4 < kDrSub / 4; ++s4) {
                const int po = (4 * s4 + c) * WS;
#pragma unroll
                for (int t = 0; t < kDrSlots; ++t) sp_dmma(acc[t], RW[(off[t] & 0xffffu) + po], W[(off[t] >> 16) + po]);
            }
        }
        double* out = p.partials + static_cast<long long>(sc) * p.svd;
#pragma unroll
        for (int t = 0; t < kDrSlots; ++t) {
            const int pair = warp * kDrSlots + t;
            if (pair < npairs) {
                const int cl = pair / ntr, tile = t0 + (pair - cl * ntr);
                *reinterpret_cast<double2*>(out + static_cast<long long>(k0 + cl) * L + tile * 64 + g * 8 + 2 * c) = make_double2(acc[t][0], acc[t][1]);
            }
        }
    }
}

}  // namespace mlb
