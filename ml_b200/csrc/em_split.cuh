// Gaussian-mixture EM, general shapes (D <= 64, K <= 256): the same feature-space formulation as the
// fused kernel of em.cu, cut into an E kernel and an M kernel because neither the parameter image
// Theta [F x K] (1.1 MB at D = 64, K = 64) nor the statistics S [F x K] fit one SM.
//
//   E kernel  (expectation_step, EM.cpp:190-219): a CTA takes a tile of 64 points, generates the feature
//             products in registers from the point tile in shared memory, and streams Theta through a
//             cp.async double buffer (L2-resident: every CTA reads the same image), one group of 32/64
//             components at a time; log-densities are stashed in shared memory, a half-warp per point does
//             the log-sum-exp, and the responsibilities go to HBM as R[point][KP] (coalesced rows).
//   M kernel  (maximisation_step, EM.cpp:221-263): work item = (chunk of points, slab of 128 features,
//             component group); the CTA re-reads the chunk's points and R rows (L2 hits across the slabs of
//             a chunk) and accumulates S = Phi^T R on the FP64 tensor pipe into registers, then writes the
//             chunk's partial statistics in the layout the fused kernel uses, so the deterministic reduction,
//             the exchange and em_finalize_kernel are shared.
// At these shapes the arithmetic intensity is > 500 flop/B, so the extra R traffic (16 KP bytes per point per
// iteration) is a few percent of the HBM time the FP64 work leaves idle (DESIGN.md "EM kernels, split path").
#pragma once

#include "fastmath.cuh"
#include "internal.h"

namespace mlb {

constexpr int kSpTile = 64;      // points per tile
constexpr int kSpThreads = 128;  // 4 warps
constexpr int kSpJB = 8;         // E-step feature steps per staged Theta block
constexpr double kLog2Pi = 0x1.d67f1c864beb4p+0;   // log(2 pi): log p(x) = log-sum-exp of the E-step terms - D/2 log(2 pi)

struct EmSplitArgs {
    const double* x;        // local points, d doubles each
    long long n_local;
    int d, k, DP, KP;
    const double* shift;    // d
    const double* theta;    // E-step image [NE][KP/16][32][2], then KP constants
    const int2* feat_e;     // [NE*4] Z-row offsets (ia, ib) of each E-step slot; (DP+1, DP+1) = unused slot
    const int2* feat_m;     // [NM*8] Z-row offsets of each M-step feature
    int ne, nm;
    double* r;              // [n_local][KP] responsibilities, a row per point
    double* partials;       // [n_chunks][sv]
    double* ll_tile;        // [n_chunks][chunk / 64]: log-likelihood sum of every 64-point tile (E kernel -> M kernel)
    int sv;
    int chunk, n_chunks;
    unsigned* counter;
    // emit
    double* r_out;          // column-major staging, leading dimension r_out_ld; scoring: log p(x) of every local point
    long long r_out_ld;
    unsigned* labels_out;
    long long range_begin, range_count;
};

__device__ __forceinline__ void sp_dmma(double (&acc)[2], double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(acc[0]), "+d"(acc[1]) : "d"(a), "d"(b));
}

__device__ __forceinline__ void sp_cp_async16(void* smem, const void* gmem)
{
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void sp_cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void sp_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// Point tile -> shared memory as z = x - shift, with the constant-1 column (0 for rows past the end) at DP and a
// zero column at DP + 1.  Columns d..DP-1 are zeroed once by the caller.
__device__ __forceinline__ void sp_load_z_tile(double* Z, int ZS, const double* x, const double* sh, long long tile0, int nvalid, int d, int DP)
{
    const double* xg = x + tile0 * d;
    const int nel = nvalid * d;
    const FastDiv by_d(d);
    // 8 loads in flight per thread before the first dependent store
    for (int e0 = threadIdx.x; e0 < kSpTile * d; e0 += 8 * kSpThreads) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * kSpThreads;
            v[u] = e < nel ? __ldg(xg + e) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int e = e0 + u * kSpThreads;
            if (e < kSpTile * d) {
                const int pt = by_d.div(e), dm = e - pt * d;
                Z[pt * ZS + dm] = e < nel ? v[u] - sh[dm] : 0.0;
            }
        }
    }
    if (threadIdx.x < kSpTile) Z[threadIdx.x * ZS + DP] = static_cast<int>(threadIdx.x) < nvalid ? 1.0 : 0.0;
}

inline size_t em_split_e_smem(int NT, int DP, int KP)
{
    return sizeof(double) * (2 * kSpJB * NT * 32 + kSpTile * (DP + 4) + kSpTile * (KP + 4) + KP + DP + kExpTableSize + 8) + sizeof(int2) * 2 * kSpJB * 4;
}

// ---------------------------------------------------------------- E kernel
// NTS = NT, or NT + kSpScore for the scoring pass, which writes log p(x) per point to r_out instead of R and the tile sums.
// (A flag inside the one int parameter keeps the names, and so the code, of the step's instances as they were.)
constexpr int kSpScore = 256;
template <int NTS>
__global__ void __launch_bounds__(kSpThreads, 2) em_split_e_kernel(const EmSplitArgs p)
{
    constexpr int NT = NTS & (kSpScore - 1);
    constexpr bool SCORE = (NTS & kSpScore) != 0;
    constexpr int KG = 8 * NT;
    extern __shared__ __align__(16) double sm[];
    const int DP = p.DP, KP = p.KP, d = p.d, ZS = DP + 4, QS = KP + 4;
    double* thS = sm;                              // [2][kSpJB][NT/2][32][2]
    double* Z = thS + 2 * kSpJB * NT * 32;         // [64][ZS]
    double* Q = Z + kSpTile * ZS;                  // [64][QS] log-densities, then responsibilities
    double* cE = Q + kSpTile * QS;                 // [KP]
    double* sh = cE + KP;                          // [DP]
    double* etab = sh + DP;                        // [32]
    double* wl = etab + kExpTableSize;             // [8]
    int2* feS = reinterpret_cast<int2*>(wl + 8);   // [2][kSpJB * 4]
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    const int ntt = KP / 8;                        // n-tiles of the whole image
    const int ngroups = KP / KG, nblocks = (p.ne + kSpJB - 1) / kSpJB;

    for (int i = tid; i < KP; i += kSpThreads) cE[i] = p.theta[static_cast<size_t>(p.ne) * ntt * 32 + i];
    for (int i = tid; i < kSpTile * ZS; i += kSpThreads) Z[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    load_exp_table(etab);

    // Stages Theta block b of component group cg (and the block's slot table) into buffer `buf`.
    auto stage = [&](int cg, int b, int buf) {
        const int j0 = b * kSpJB;
        const int nj = min(kSpJB, p.ne - j0);
        double* dst = thS + buf * (kSpJB * NT * 32);
        // per step: NT * 32 doubles = NT * 16 chunks of 16 bytes, contiguous in the image
        for (int i = tid; i < nj * NT * 16; i += kSpThreads) {
            const int jj = i / (NT * 16), q = i - jj * (NT * 16);
            const double* src = p.theta + (static_cast<size_t>(j0 + jj) * ntt + cg * NT) * 32 + q * 2;
            sp_cp_async16(dst + jj * NT * 32 + q * 2, src);
        }
        int2* fdst = feS + buf * (kSpJB * 4);
        for (int i = tid; i < nj * 2; i += kSpThreads) sp_cp_async16(fdst + i * 2, p.feat_e + j0 * 4 + i * 2);
        sp_cp_async_commit();
    };

    // Work item = one 64-point tile (chunks are multiples of 128 points, so tiles never straddle a chunk): fine enough
    // to balance 148 SMs whatever the chunk size.  The tile's log-likelihood sum goes to ll_tile; the M kernel adds the
    // tiles of a chunk in order into the chunk's partial.
    const int tpc = p.chunk / kSpTile;
    const int nitems = p.n_chunks * tpc;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int item = s_next;
        if (item >= nitems) break;
        const int chunk = item / tpc, t = item - chunk * tpc;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const long long p_end = p_begin + p.chunk < p.n_local ? p_begin + p.chunk : p.n_local;
        double ll_acc = 0.0, ll_prod = 1.0;
        {
            const long long tile0 = p_begin + static_cast<long long>(t) * kSpTile;
            if (tile0 >= p_end) {
                if (!SCORE && tid == 0) p.ll_tile[item] = 0.0;
                continue;
            }
            const int nvalid = static_cast<int>(p_end - tile0 < kSpTile ? p_end - tile0 : kSpTile);
            sp_load_z_tile(Z, ZS, p.x, sh, tile0, nvalid, d, DP);
            const double* z0 = Z + (warp * 16 + g) * ZS;
            const double* z1 = z0 + 8 * ZS;
            for (int cg = 0; cg < ngroups; ++cg) {
                double acc[2][NT][2];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) acc[0][nt][0] = acc[0][nt][1] = acc[1][nt][0] = acc[1][nt][1] = 0.0;
                stage(cg, 0, 0);
                for (int b = 0; b < nblocks; ++b) {
                    if (b + 1 < nblocks) {
                        stage(cg, b + 1, (b + 1) & 1);
                        sp_cp_async_wait<1>();
                    } else {
                        sp_cp_async_wait<0>();
                    }
                    __syncthreads();
                    const double* th = thS + (b & 1) * (kSpJB * NT * 32);
                    const int2* fe = feS + (b & 1) * (kSpJB * 4);
                    const int nj = min(kSpJB, p.ne - b * kSpJB);
#pragma unroll 4
                    for (int jj = 0; jj < nj; ++jj) {
                        const int2 f = fe[jj * 4 + c];
                        const double a0 = z0[f.x] * z0[f.y], a1 = z1[f.x] * z1[f.y];
#pragma unroll
                        for (int h = 0; h < NT / 2; ++h) {
                            const double2 bb = reinterpret_cast<const double2*>(th)[(jj * (NT / 2) + h) * 32 + lane];
                            sp_dmma(acc[0][2 * h], a0, bb.x);
                            sp_dmma(acc[1][2 * h], a1, bb.x);
                            sp_dmma(acc[0][2 * h + 1], a0, bb.y);
                            sp_dmma(acc[1][2 * h + 1], a1, bb.y);
                        }
                    }
                    __syncthreads();   // the buffer is refilled two blocks later
                }
                // stash the group's log-densities (plus the per-component constant)
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    double* qrow = Q + (warp * 16 + mt * 8 + g) * QS + cg * KG;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        const int kk = 8 * nt + 2 * c;
                        const double2 cc = *reinterpret_cast<const double2*>(cE + cg * KG + kk);
                        *reinterpret_cast<double2*>(qrow + kk) = make_double2(acc[mt][nt][0] + cc.x, acc[mt][nt][1] + cc.y);
                    }
                }
            }
            __syncwarp();
            // ---------------- log-sum-exp: a half-warp per point, 8 passes over the warp's 16 points
            const int hl = lane & 15;
            for (int pass = 0; pass < 8; ++pass) {
                const int pl = warp * 16 + pass * 2 + (lane >> 4);
                double* qrow = Q + pl * QS;
                double mx = -INFINITY;
                for (int kk = hl; kk < KP; kk += 16) mx = fmax(mx, qrow[kk]);
#pragma unroll
                for (int off = 8; off >= 1; off >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                double sum = 0.0;
                for (int kk = hl; kk < KP; kk += 16) {
                    const double e = exp_nonpositive(qrow[kk] - mx, etab);
                    if (!SCORE) qrow[kk] = e;
                    sum += e;
                }
#pragma unroll
                for (int off = 8; off >= 1; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
                if constexpr (SCORE) {
                    if (pl < nvalid && hl == 0) p.r_out[tile0 + pl] = (mx + log(sum)) - 0.5 * d * kLog2Pi;
                    continue;
                }
                const double inv = reciprocal_of_sum(sum);
                if (pl < nvalid) {
                    double* rrow = p.r + (tile0 + pl) * KP;
                    for (int kk = hl; kk < KP; kk += 16) rrow[kk] = qrow[kk] * inv;
                    if (hl == 0) {
                        ll_acc += mx;
                        ll_prod *= sum;
                    }
                }
            }
            ll_acc += log(ll_prod);
        }
        if constexpr (SCORE) {
            __syncthreads();   // Z and Q are rewritten by the next item
            continue;
        }

        // log-likelihood sum of the tile: fixed butterfly inside the warp, fixed order across warps
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) ll_acc += __shfl_xor_sync(0xffffffffu, ll_acc, off);
        if (lane == 0) wl[warp] = ll_acc;
        __syncthreads();   // also: Z and Q are rewritten by the next item
        if (tid == 0) p.ll_tile[item] = (wl[0] + wl[1]) + (wl[2] + wl[3]);
    }
}

constexpr int kSpTileM = 32;     // points per M-step tile (double-buffered with cp.async)

inline size_t em_split_m_smem(int NW, int DP)
{
    return sizeof(double) * (2 * kSpTileM * (DP + 4) + 2 * kSpTileM * (8 * NW + 4) + DP);
}

__device__ __forceinline__ void sp_cp_async8(void* smem, const void* gmem)
{
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem));
}

// ---------------------------------------------------------------- M kernel
// MW = feature tiles (of 8) per warp: a CTA covers 4 * MW * 8 features of one slab; the host picks the MW in {3, 4, 5}
// that wastes the fewest tile slots for the shape (D = 16: 5, one slab; D = 32: 3; D = 64: 4).
template <int NW, int MW>
__global__ void __launch_bounds__(kSpThreads, (NW * MW > 32) ? 1 : 2) em_split_m_kernel(const EmSplitArgs p)
{
    constexpr int KG = 8 * NW, RS = KG + 4, TM = kSpTileM;
    extern __shared__ __align__(16) double sm[];
    const int DP = p.DP, KP = p.KP, d = p.d, ZS = DP + 4;
    double* Zb = sm;                        // [2][TM][ZS]
    double* Rb = Zb + 2 * TM * ZS;          // [2][TM][RS]
    double* sh = Rb + 2 * TM * RS;          // [DP]
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    const int ngroups = KP / KG;
    const int nslabs = (p.nm + 4 * MW - 1) / (4 * MW);
    const int nitems = p.n_chunks * nslabs * ngroups;
    const FastDiv by_d(d);

    for (int i = tid; i < 2 * TM * ZS; i += kSpThreads) Zb[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int item = s_next;
        if (item >= nitems) break;
        // consecutive items share a chunk, so concurrently running CTAs re-read the same points and R rows from L2
        const int chunk = item / (nslabs * ngroups);
        const int rem = item - chunk * (nslabs * ngroups);
        const int slab = rem / ngroups, cg = rem - slab * ngroups;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const long long p_end = p_begin + p.chunk < p.n_local ? p_begin + p.chunk : p.n_local;
        const int ntiles = static_cast<int>((p_end - p_begin + TM - 1) / TM);

        // Asynchronous copy of the raw coordinates and the R rows of one tile; rows past the end are zeroed.
        auto stage = [&](int t, int buf) {
            const long long tile0 = p_begin + static_cast<long long>(t) * TM;
            const int nvalid = static_cast<int>(p_end - tile0 < TM ? p_end - tile0 : TM);
            double* Z = Zb + buf * (TM * ZS);
            double* R = Rb + buf * (TM * RS);
            const double* xg = p.x + tile0 * d;
            const int nel = nvalid * d;
            if ((d & 1) == 0) {
                // even dimension: rows are 16-byte aligned on both sides, two coordinates per copy
                const int hd = d >> 1;
                const FastDiv by_hd(hd);
                for (int e2 = tid; e2 < TM * hd; e2 += kSpThreads) {
                    const int pt = by_hd.div(e2), q = e2 - pt * hd;
                    if (2 * e2 < nel) sp_cp_async16(Z + pt * ZS + 2 * q, xg + 2 * e2);
                    else *reinterpret_cast<double2*>(Z + pt * ZS + 2 * q) = make_double2(0.0, 0.0);
                }
            } else {
                for (int e = tid; e < TM * d; e += kSpThreads) {
                    const int pt = by_d.div(e), dm = e - pt * d;
                    if (e < nel) sp_cp_async8(Z + pt * ZS + dm, xg + e);
                    else Z[pt * ZS + dm] = 0.0;
                }
            }
            for (int e = tid; e < TM * (KG / 2); e += kSpThreads) {
                const int pt = e / (KG / 2), q = e - pt * (KG / 2);
                if (pt < nvalid) sp_cp_async16(R + pt * RS + 2 * q, p.r + (tile0 + pt) * KP + cg * KG + 2 * q);
                else *reinterpret_cast<double2*>(R + pt * RS + 2 * q) = make_double2(0.0, 0.0);
            }
            sp_cp_async_commit();
        };
        // Each thread shifts the coordinates it copied itself (visible to it after its own wait), then the block syncs.
        auto finish = [&](int t, int buf) {
            const long long tile0 = p_begin + static_cast<long long>(t) * TM;
            const int nvalid = static_cast<int>(p_end - tile0 < TM ? p_end - tile0 : TM);
            double* Z = Zb + buf * (TM * ZS);
            const int nel = nvalid * d;
            if ((d & 1) == 0) {
                const int hd = d >> 1;
                const FastDiv by_hd(hd);
                for (int e2 = tid; 2 * e2 < nel; e2 += kSpThreads) {
                    const int pt = by_hd.div(e2), q = e2 - pt * hd;
                    double2* cell = reinterpret_cast<double2*>(Z + pt * ZS + 2 * q);
                    const double2 v = *cell;
                    *cell = make_double2(v.x - sh[2 * q], v.y - sh[2 * q + 1]);
                }
            } else {
                for (int e = tid; e < nel; e += kSpThreads) {
                    const int pt = by_d.div(e), dm = e - pt * d;
                    Z[pt * ZS + dm] -= sh[dm];
                }
            }
            if (tid < TM) Z[tid * ZS + DP] = tid < nvalid ? 1.0 : 0.0;
        };

        int ia[MW], ib[MW];
#pragma unroll
        for (int i = 0; i < MW; ++i) {
            const int mt = (slab * 4 + warp) * MW + i;
            const int2 f = mt < p.nm ? p.feat_m[mt * 8 + g] : make_int2(DP + 1, DP + 1);
            ia[i] = f.x;
            ib[i] = f.y;
        }
        double acc[MW][NW][2];
#pragma unroll
        for (int i = 0; i < MW; ++i)
#pragma unroll
            for (int nt = 0; nt < NW; ++nt) acc[i][nt][0] = acc[i][nt][1] = 0.0;

        stage(0, 0);
        for (int t = 0; t < ntiles; ++t) {
            if (t + 1 < ntiles) {
                stage(t + 1, (t + 1) & 1);
                sp_cp_async_wait<1>();
            } else {
                sp_cp_async_wait<0>();
            }
            finish(t, t & 1);
            __syncthreads();
            const double* Z = Zb + (t & 1) * (TM * ZS);
            const double* R = Rb + (t & 1) * (TM * RS);
#pragma unroll 2
            for (int s = 0; s < TM / 4; ++s) {
                const double* zp = Z + (4 * s + c) * ZS;
                const double* rp = R + (4 * s + c) * RS + g;
                double bf[NW];
#pragma unroll
                for (int nt = 0; nt < NW; ++nt) bf[nt] = rp[8 * nt];
#pragma unroll
                for (int i = 0; i < MW; ++i) {
                    const double af = zp[ia[i]] * zp[ib[i]];
#pragma unroll
                    for (int nt = 0; nt < NW; ++nt) sp_dmma(acc[i][nt], af, bf[nt]);
                }
            }
            __syncthreads();   // the buffer is refilled by the stage() of the next iteration
        }

        double* out = p.partials + static_cast<long long>(chunk) * p.sv;
        if (slab == 0 && cg == 0 && tid < 8) {
            // the chunk's log-likelihood partial: its tiles' sums (E kernel) added in tile order
            double ll = 0.0;
            if (tid == 0) {
                const int tpc = p.chunk / kSpTile;
                for (int t = 0; t < tpc; ++t) ll += p.ll_tile[static_cast<long long>(chunk) * tpc + t];
            }
            out[p.sv - 8 + tid] = ll;
        }
#pragma unroll
        for (int i = 0; i < MW; ++i) {
            const int mt = (slab * 4 + warp) * MW + i;
            if (mt < p.nm) {
#pragma unroll
                for (int nt = 0; nt < NW; ++nt)
                    *reinterpret_cast<double2*>(out + static_cast<long long>(mt * 8 + g) * KP + cg * KG + nt * 8 + 2 * c) = make_double2(acc[i][nt][0], acc[i][nt][1]);
            }
        }
    }
}

// ---------------------------------------------------------------- emit: R rows -> column-major staging + labels
// responsibilities_ (EM.cpp:213-218) and labels_ (EM.cpp:289-304: argmax, first maximum wins; a NaN row gives UINT_MAX).
__global__ void em_split_emit_kernel(const EmSplitArgs p)
{
    __shared__ double T[32][33];
    const long long row0 = p.range_begin + static_cast<long long>(blockIdx.x) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    const long long hi = p.range_begin + p.range_count;
    if (p.r_out) {
        for (int k0 = 0; k0 < p.k; k0 += 32) {
            for (int i = ty; i < 32; i += 8) {
                const long long pt = row0 + i;
                T[i][tx] = (pt < hi && k0 + tx < p.k) ? p.r[pt * p.KP + k0 + tx] : 0.0;
            }
            __syncthreads();
            for (int i = ty; i < 32; i += 8) {
                const long long pt = row0 + tx;
                if (pt < hi && k0 + i < p.k) p.r_out[(pt - p.range_begin) + static_cast<long long>(k0 + i) * p.r_out_ld] = T[tx][i];
            }
            __syncthreads();
        }
    }
    if (p.labels_out && ty == 0) {
        const long long pt = row0 + tx;
        if (pt < hi) {
            const double* rrow = p.r + pt * p.KP;
            double best = -1.0;
            unsigned best_k = 0xffffffffu;
            for (int kk = 0; kk < p.k; ++kk) {
                const double r = rrow[kk];
                if (r > best) { best = r; best_k = static_cast<unsigned>(kk); }
            }
            p.labels_out[pt - p.range_begin] = best_k;
        }
    }
}

// Host responsibilities (column-major n x k, already on the device) -> R rows, padded components zero.
__global__ void em_split_import_r_kernel(const double* r_in, long long ld, long long n, int k, int KP, double* r)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n * KP) return;
    const long long pt = i / KP;
    const int kk = static_cast<int>(i - pt * KP);
    r[i] = kk < k ? r_in[pt + kk * ld] : 0.0;
}

}  // namespace mlb
